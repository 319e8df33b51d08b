// Connected components of a graph given as a bit adjacency matrix, or of a node's proper-cluster graph given
// by its leaf tours (tour_components_async: no graph needed).
//
// Replaces _get_graph_components of the reference (/root/reference/src/sc_supertree/scs.py:458-492).
// The reference explores the `edges` sets, i.e. "the pair co-occurred in some tree", which is the
// adjacency bit matrix the row kernel emits (C > 0), not W > 0.
//
// Lock-free union-find.  Roots are always hooked larger-under-smaller, so the final root of a
// component is its smallest vertex id whatever the interleaving -- labels are deterministic.
// The graphs here are dense (10^7 .. 10^8 set bits at 10^4 vertices) and usually one giant
// component, so hooking every edge would be per-bit work for nothing.  Sampling first, as in
// Afforest (Sutton et al.): (1) every vertex is hooked to its first two neighbours only;
// (2) the trees are flattened and the most frequent root among 1024 sampled vertices is taken as the
// giant component; (3) only the rows of vertices OUTSIDE the giant are hooked in full (all their
// neighbours, smaller ids too: the adjacency is symmetric, so every edge with an endpoint outside the
// giant is seen from that endpoint, and edges inside it change nothing).

#include "common.cuh"
#include "uf.cuh"

namespace scs {

namespace {

__global__ void uf_init(int n, int32_t *parent) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) parent[i] = i;
}

// (1) one warp per row: hook the vertex to its first kSample neighbours
constexpr int kSample = 2;
__global__ void uf_hook_sample(int n, int words, const uint32_t *__restrict__ bits, int32_t *parent) {
    const int warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp_global >= n) return;
    const int a = warp_global;
    const uint32_t *row = bits + static_cast<size_t>(a) * words;
    int found = 0;
    for (int j0 = 0; j0 < words && found < kSample; j0 += 32) {
        const int j = j0 + lane;
        uint32_t wbits = j < words ? row[j] : 0u;
        if (j == (a >> 5)) wbits &= ~(1u << (a & 31));
        unsigned active = __ballot_sync(0xffffffffu, wbits != 0u);
        while (active && found < kSample) {
            const int src = __ffs(active) - 1;
            uint32_t wsrc = __shfl_sync(0xffffffffu, wbits, src);
            while (wsrc && found < kSample) {
                const int b = ((j0 + src) << 5) + __ffs(wsrc) - 1;
                wsrc &= wsrc - 1;
                if (b < n) {
                    if (lane == 0) uf_union(parent, a, b);
                    ++found;
                }
            }
            active &= active - 1;
        }
    }
}

// (2a) flatten: snapshot[i] = root of i (the forest only changes at roots afterwards)
__global__ void uf_snapshot(int n, int32_t *parent, int32_t *snapshot) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int r = i;
    while (parent[r] != r) r = parent[r];
    snapshot[i] = r;
}

// (2b) the most frequent root among up to 1024 evenly spaced vertices; one CTA of 1024 threads
__global__ void __launch_bounds__(1024) uf_pick_giant(int n, const int32_t *__restrict__ snapshot, int32_t *giant) {
    __shared__ int32_t roots[1024];
    __shared__ int best_count[32];
    __shared__ int32_t best_root[32];
    const int tid = threadIdx.x;
    const int samples = n < 1024 ? n : 1024;
    const int32_t mine = tid < samples ? snapshot[static_cast<int64_t>(tid) * n / samples] : -1;
    roots[tid] = mine;
    __syncthreads();
    int count = 0;
    if (mine >= 0)
        for (int i = 0; i < samples; ++i) count += roots[i] == mine;
    int32_t root = mine;
    for (int off = 16; off > 0; off >>= 1) {
        const int oc = __shfl_down_sync(0xffffffffu, count, off);
        const int32_t orr = __shfl_down_sync(0xffffffffu, root, off);
        if (oc > count || (oc == count && orr >= 0 && (root < 0 || orr < root))) { count = oc; root = orr; }
    }
    if ((tid & 31) == 0) { best_count[tid >> 5] = count; best_root[tid >> 5] = root; }
    __syncthreads();
    if (tid == 0) {
        int bc = best_count[0];
        int32_t br = best_root[0];
        for (int w = 1; w < 32; ++w)
            if (best_count[w] > bc || (best_count[w] == bc && best_root[w] >= 0 && (br < 0 || best_root[w] < br))) {
                bc = best_count[w];
                br = best_root[w];
            }
        *giant = br;
    }
}

// (3) one warp per row outside the giant component; lanes take words of the row, every neighbour is hooked
__global__ void uf_hook_rest(int n, int words, const uint32_t *__restrict__ bits, const int32_t *__restrict__ snapshot,
                             const int32_t *__restrict__ giant, int32_t *parent) {
    const int warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp_global >= n) return;
    const int a = warp_global;
    if (snapshot[a] == *giant) return;
    const uint32_t *row = bits + static_cast<size_t>(a) * words;
    for (int j = lane; j < words; j += 32) {
        uint32_t wbits = row[j];
        const int first = j << 5;
        if (j == (a >> 5)) wbits &= ~(1u << (a & 31));
        while (wbits) {
            const int b = first + __ffs(wbits) - 1;
            wbits &= wbits - 1;
            if (b < n) uf_union(parent, a, b);
        }
    }
}

__global__ void uf_flatten(int n, int32_t *parent, int32_t *label, int32_t *n_roots) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int r = i;
    while (parent[r] != r) r = parent[r];
    label[i] = r;
    if (r == i) atomicAdd(n_roots, 1);
}

// Components straight from the leaf tours.  Taxa a and b are adjacent iff some tree holds both with their
// LCA below its root; the leaves under one child of a root are a contiguous run of the tour whose
// consecutive LCAs all lie below the root.  So hooking every consecutive pair i, i + 1 of a tree whose
// adj_depth differs from the tree's root depth (the root test of the graph build) yields the same
// components.  One thread per tour entry.  As on the bits, hooking every pair of a giant component is contention for
// nothing: a first launch hooks every kTourSample-th pair only (snapshot == nullptr), then the roots are
// snapshotted and the second launch hooks only the pairs whose snapshot roots still differ.
constexpr int kTourSample = 16;
__global__ void uf_hook_tours(int n, int T, int64_t L, const int64_t *__restrict__ leaf_offsets,
                              const int32_t *__restrict__ leaf_taxon, const int32_t *__restrict__ adj_depth,
                              const int32_t *__restrict__ root_depth, const int32_t *__restrict__ snapshot,
                              int32_t *parent, int32_t *__restrict__ bad) {
    const int64_t g = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
    if (g >= L || (!snapshot && g % kTourSample != 0)) return;
    int lo = 0, hi = T;  // largest t with leaf_offsets[t] <= g
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (leaf_offsets[mid] <= g) lo = mid; else hi = mid;
    }
    const int64_t end = leaf_offsets[lo + 1];
    const int a = leaf_taxon[g];
    // out of range, or more leaves than taxa (a repeated taxon): rejected like the graph build rejects it
    if (a < 0 || a >= n || end - leaf_offsets[lo] > n) { *bad = 1; return; }
    if (g + 1 >= end || adj_depth[g] == root_depth[lo]) return;
    const int b = leaf_taxon[g + 1];
    if (b < 0 || b >= n || (snapshot && snapshot[a] == snapshot[b])) return;
    uf_union(parent, a, b);
}

}  // namespace

// Enqueue only: label[v] = smallest vertex of v's component, *count_dev = number of components.
int components_async(scs_ctx *ctx, int n, const uint32_t *bits, int32_t *label, int32_t *count_dev) {
    if (n <= 0 || !bits || !label || !count_dev) return fail(ctx, SCS_ERR_INVALID, "components: bad argument");
    const int words = scs_bit_words(n);
    int32_t *parent;
    int rc;
    // the union-find forest is built in `label` itself, then flattened in place
    if ((rc = reserve_as(ctx, SLOT_UF_PARENT, static_cast<size_t>(n), &parent))) return rc;
    SCS_CUDA(ctx, cudaMemsetAsync(count_dev, 0, sizeof(int32_t), ctx->stream));
    uf_init<<<ceil_div(n, 256), 256, 0, ctx->stream>>>(n, parent);
    SCS_LAUNCHED(ctx, "uf_init");
    const int row_blocks = ceil_div(static_cast<int64_t>(n) * 32, 256);
    int32_t *giant = count_dev + 4;  // scratch next to the counter (scalars slot)
    uf_hook_sample<<<row_blocks, 256, 0, ctx->stream>>>(n, words, bits, parent);
    SCS_LAUNCHED(ctx, "uf_hook_sample");
    uf_snapshot<<<ceil_div(n, 256), 256, 0, ctx->stream>>>(n, parent, label);
    SCS_LAUNCHED(ctx, "uf_snapshot");
    uf_pick_giant<<<1, 1024, 0, ctx->stream>>>(n, label, giant);
    SCS_LAUNCHED(ctx, "uf_pick_giant");
    uf_hook_rest<<<row_blocks, 256, 0, ctx->stream>>>(n, words, bits, label, giant, parent);
    SCS_LAUNCHED(ctx, "uf_hook_rest");
    uf_flatten<<<ceil_div(n, 256), 256, 0, ctx->stream>>>(n, parent, label, count_dev);
    SCS_LAUNCHED(ctx, "uf_flatten");
    return SCS_OK;
}

// Enqueue only: the components of the node's proper-cluster graph from its tours, labelled as components_async
// labels them; *bad_dev is raised for a malformed tour.  Neither counter is cleared here.
int tour_components_async(scs_ctx *ctx, int n, int T, int64_t L, const int64_t *leaf_offsets,
                          const int32_t *leaf_taxon, const int32_t *adj_depth, const int32_t *root_depth,
                          int32_t *label, int32_t *count_dev, int32_t *bad_dev) {
    if (n <= 0 || T < 0 || L < 0 || !label || !count_dev || !bad_dev)
        return fail(ctx, SCS_ERR_INVALID, "tour components: bad argument");
    int32_t *parent;
    int rc;
    if ((rc = reserve_as(ctx, SLOT_UF_PARENT, static_cast<size_t>(n), &parent))) return rc;
    uf_init<<<ceil_div(n, 256), 256, 0, ctx->stream>>>(n, parent);
    SCS_LAUNCHED(ctx, "uf_init");
    if (L > 0 && T > 0) {
        // the snapshot lives in `label` until the final flatten overwrites it
        uf_hook_tours<<<ceil_div(L, 256), 256, 0, ctx->stream>>>(n, T, L, leaf_offsets, leaf_taxon, adj_depth,
                                                                 root_depth, nullptr, parent, bad_dev);
        SCS_LAUNCHED(ctx, "uf_hook_tours");
        uf_snapshot<<<ceil_div(n, 256), 256, 0, ctx->stream>>>(n, parent, label);
        SCS_LAUNCHED(ctx, "uf_snapshot");
        uf_hook_tours<<<ceil_div(L, 256), 256, 0, ctx->stream>>>(n, T, L, leaf_offsets, leaf_taxon, adj_depth,
                                                                 root_depth, label, parent, bad_dev);
        SCS_LAUNCHED(ctx, "uf_hook_tours");
    }
    uf_flatten<<<ceil_div(n, 256), 256, 0, ctx->stream>>>(n, parent, label, count_dev);
    SCS_LAUNCHED(ctx, "uf_flatten");
    return SCS_OK;
}

int components(scs_ctx *ctx, int n, const uint32_t *bits, int32_t *label, int32_t *n_components_host) {
    int32_t *scalars;
    int rc;
    if ((rc = reserve_as(ctx, SLOT_SCALARS, 64, &scalars))) return rc;
    int32_t *n_roots = scalars + 8;
    if ((rc = components_async(ctx, n, bits, label, n_roots))) return rc;
    if (n_components_host) {
        void *pin;
        if ((rc = reserve_pinned(ctx, 64, &pin))) return rc;
        SCS_CUDA(ctx, cudaMemcpyAsync(pin, n_roots, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        *n_components_host = *static_cast<int32_t *>(pin);
    }
    return SCS_OK;
}

}  // namespace scs
