// Device-resident source trees: upload, leaf tours, restriction to the children of a wave (see devforest.cuh).
//
// Restriction.  The reference restricts every source tree to the taxa of a component with
// PhyloNode.get_sub_tree(names, ignore_missing=True, as_rooted=True) (/root/reference/src/sc_supertree/scs.py:444-453);
// forest.cpp does the same on flat arrays on the host, one linear pass per (tree, child).  Here a (tree, child) pair is
// walked by a warp, or by a whole CTA when its tree is large, and the passes are prefix sums over the tree's pre-order
// node array:
//   kept[k]     tip whose taxon belongs to the child;           P = exclusive prefix sum of kept
//   cnt[k]      kept tips below k = P[k + size[k]] - P[k]       (pre-order: a subtree is a contiguous run)
//   unary[k]    some child of k carries all of cnt[k]           (set by that child: cnt[child] == cnt[k])
//   retained[k] cnt[k] > 0 and (tip or not unary[k]);           R = exclusive prefix sum of retained = new index
// A retained node then walks up its chain of merged (unary) ancestors, folding their lengths bottom-up in the
// reference's operand order  length(node) + length(child)  -- the same additions in the same order as forest.cpp and
// tree.py, so branch-length weights stay bit-identical at every recursion level.  The first retained node in
// pre-order is the new root and loses its length.  Which (tree, child) pairs exist (>= 2 kept tips, scs.py:447-448)
// comes from a histogram of the tips over the children, scanned into a dense pair list ordered by child, then tree:
// the new forest is laid out by child with its trees in source order (the graph build sums W in tree input order).

#include "devforest.cuh"

#include <algorithm>
#include <cmath>
#include <cstddef>
#include <cstdlib>
#include <vector>

#include <omp.h>

#include "forest.hpp"
#include "shard.cuh"

namespace scs {

int grow(scs_ctx *ctx, GrowBuf &buf, size_t bytes) {
    if (bytes == 0) bytes = 16;
    if (buf.bytes >= bytes) return SCS_OK;
    const size_t want = bytes + bytes / 4 + 256;
    if (buf.ptr) {
        SCS_CUDA(ctx, cudaFreeAsync(buf.ptr, ctx->stream));
        buf.ptr = nullptr;
        buf.bytes = 0;
    }
    const cudaError_t err = cudaMallocAsync(&buf.ptr, want, ctx->stream);
    if (err != cudaSuccess) {
        buf.ptr = nullptr;
        return fail(ctx, SCS_ERR_CUDA, "cudaMallocAsync (device forest)", err);
    }
    buf.bytes = want;
    return SCS_OK;
}

void release(scs_ctx *ctx, GrowBuf &buf) {
    if (buf.ptr) cudaFreeAsync(buf.ptr, ctx->stream);
    buf.ptr = nullptr;
    buf.bytes = 0;
}

void DevForest::free_all(scs_ctx *ctx) {
    for (GrowBuf *b : {&tree_off, &leaf_off, &parent, &size, &taxon, &length, &support, &weight, &tree_job}) release(ctx, *b);
    trees = nodes = leaves = 0;
}

void DevTours::free_all(scs_ctx *ctx) {
    for (GrowBuf *b : {&leaf_taxon, &adj_depth, &root_depth, &adj_val, &depth_s, &val_s}) release(ctx, *b);
}

namespace {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kBlock = 256;  // threads of every tour and restriction launch
constexpr int kWarps = kBlock / 32;
// A tree (tours) or a (tree, part) pair (restriction) of more nodes than this is walked by a whole CTA, in chunks of
// kBlock * kChunkItems pre-order nodes; a smaller one by a warp, 32 nodes at a time.  Measured on C4, profiles/README.md.
constexpr int kCtaNodes = 256;
constexpr int kChunkItems = 4;

__device__ __forceinline__ int warp_excl_scan(int v, int lane, int &total) {
    int inc = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int o = __shfl_up_sync(kFull, inc, off);
        if (lane >= off) inc += o;
    }
    total = __shfl_sync(kFull, inc, 31);
    return inc - v;
}

// The threads that walk one tree: a warp, or the whole CTA.  A thread holds kItems consecutive nodes of a chunk;
// excl_scan is the exclusive prefix sum over the group in rank order, plus the group's total.
struct WarpGroup {
    static constexpr int kSize = 32, kItems = 1;
    int rank;
    __device__ void sync() const { __syncwarp(); }
    __device__ int excl_scan(int v, int &total) const { return warp_excl_scan(v, rank, total); }
};

struct BlockGroup {
    static constexpr int kSize = kBlock, kItems = kChunkItems;
    int rank;
    int *warp_sum;  // shared [kWarps]
    __device__ void sync() const { __syncthreads(); }
    __device__ int excl_scan(int v, int &total) const {
        const int lane = rank & 31, warp = rank >> 5;
        int wt;
        const int e = warp_excl_scan(v, lane, wt);
        if (lane == 0) warp_sum[warp] = wt;
        __syncthreads();
        int before = 0, all = 0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) {
            const int s = warp_sum[w];
            before += w < warp ? s : 0;
            all += s;
        }
        __syncthreads();  // warp_sum is rewritten by the next scan
        total = all;
        return before + e;
    }
};

// Items [0, n) -- trees or pairs -- over the grid.  Block b walks the large items i = b (mod blocks) one after the other
// with all its threads; then every warp of the grid takes the small items i = w (mod warps).  The grid is sized on the
// host from a bound of n: n itself may live on the device.
template <class Large, class OnBlock, class OnWarp>
__device__ void for_each_item(int n, Large large, OnBlock on_block, OnWarp on_warp) {
    __shared__ int list[kBlock];
    __shared__ int listed;
    const int64_t G = gridDim.x;
    for (int64_t r0 = blockIdx.x; r0 < n; r0 += G * kBlock) {
        if (threadIdx.x == 0) listed = 0;
        __syncthreads();
        const int64_t i = r0 + G * threadIdx.x;
        if (i < n && large(static_cast<int>(i))) list[atomicAdd(&listed, 1)] = static_cast<int>(i);
        __syncthreads();
        const int m = listed;
        for (int j = 0; j < m; ++j) on_block(list[j]);
        __syncthreads();  // list and listed are rewritten by the next round
    }
    const int64_t warps = G * kWarps;
    for (int64_t i = blockIdx.x * static_cast<int64_t>(kWarps) + (threadIdx.x >> 5); i < n; i += warps)
        if (!large(static_cast<int>(i))) on_warp(static_cast<int>(i));
}

// ---- tours (scs.py:555-567, 628: the value handed top-down; forest.cpp:scs_forest_tours) -----------------------------
// Pass A: depth and weighting value of every internal node, top-down, a chunk of pre-order nodes at a time; a node whose
// parent sits in the same chunk waits for it (parents come first in pre-order, so some waiting node is always ready).
// Every value is  value(parent) + own  in that operand order: the sums of forest.cpp, bit for bit.  Pass B: every tip
// writes its tour entry, numbered by a prefix sum over the tips.
struct TourArgs {
    const int64_t *tree_off, *leaf_off;
    const int32_t *parent, *taxon;
    const double *length, *support;
    int weighting;
    const int32_t *taxon_vertex;
    int32_t *depth_s;
    double *val_s;
    int32_t *leaf_taxon, *adj_depth;
    double *adj_val;
    int32_t *root_depth, *flags;
};

__device__ __forceinline__ double own_value(const TourArgs &a, int64_t node) {  // an internal node below the root
    if (a.weighting == 1) {
        const double len = a.length[node];
        return isnan(len) ? 1.0 : len;
    }
    return a.weighting == 3 ? a.support[node] : 0.0;
}

__device__ __forceinline__ double value_below(int weighting, double above, double own) {
    switch (weighting) {
    case 0: return 1.0;
    case 1: return above + own;
    case 2: return above + 1.0;
    default: return own;
    }
}

// tour entry pos of tip k of the tree at base
__device__ __forceinline__ void write_tip(const TourArgs &a, int64_t base, int count, int k, int64_t pos) {
    a.leaf_taxon[pos] = a.taxon_vertex[a.taxon[base + k]];
    if (k + 1 < count) {
        const int lca = a.parent[base + k + 1];  // the next pre-order node hangs off the LCA with the next tip
        const double x = a.val_s[base + lca];
        a.adj_depth[pos] = a.depth_s[base + lca];
        a.adj_val[pos] = x;
        if (lca != 0 && isnan(x)) a.flags[1] = 1;  // bootstrap weighting without a support value
    } else {
        a.adj_depth[pos] = -1;
        a.adj_val[pos] = 0.0;
    }
}

// a small tree: one warp, 32 nodes per chunk; waiting nodes take their parent's value by shuffle
__device__ void tours_warp(const TourArgs &a, int t, int lane) {
    const int64_t base = a.tree_off[t];
    const int count = static_cast<int>(a.tree_off[t + 1] - base);
    if (lane == 0) a.root_depth[t] = 0;
    if (count <= 1) return;  // a lone tip has no sides (scs.py:570)
    const int32_t *par = a.parent + base;
    const int32_t *tax = a.taxon + base;
    for (int c0 = 0; c0 < count; c0 += 32) {
        const int k = c0 + lane;
        const bool internal = k < count && tax[k] < 0;
        const int p = internal && k > 0 ? par[k] : 0;
        const double own = internal && k > 0 ? own_value(a, base + k) : 0.0;
        double v = 0.0;  // the value handed to the root's children is 0 (scs.py:577)
        int d = 0;
        bool pending = internal && k > 0;
        if (pending && p < c0) {
            v = value_below(a.weighting, a.val_s[base + p], own);
            d = a.depth_s[base + p] + 1;
            pending = false;
        }
        unsigned waiting = __ballot_sync(kFull, pending);
        while (waiting) {
            const int src = pending ? p - c0 : 0;
            const double above = __shfl_sync(kFull, v, src);
            const int dabove = __shfl_sync(kFull, d, src);
            if (pending && !((waiting >> src) & 1u)) {
                v = value_below(a.weighting, above, own);
                d = dabove + 1;
                pending = false;
            }
            waiting = __ballot_sync(kFull, pending);
        }
        if (internal) {
            a.val_s[base + k] = v;
            a.depth_s[base + k] = d;
        }
        __syncwarp();
    }
    const int64_t o = a.leaf_off[t];
    int tip_base = 0;
    for (int c0 = 0; c0 < count; c0 += 32) {
        const int k = c0 + lane;
        const bool tip = k < count && tax[k] >= 0;
        const unsigned tips = __ballot_sync(kFull, tip);
        if (tip) write_tip(a, base, count, k, o + tip_base + __popc(tips & ((1u << lane) - 1u)));
        tip_base += __popc(tips);
    }
}

constexpr int kTourChunk = kBlock * kChunkItems;
struct TourShared {
    double val[kTourChunk];
    int32_t depth[kTourChunk];
    int32_t stamp[kTourChunk];  // 0: pending; r: resolved before the barrier that opened round r (or by this thread)
};

// a large tree: the whole CTA, kTourChunk nodes per chunk.  Waiting nodes resolve in rounds separated by block
// barriers; a thread also resolves, within a round, a node whose parent is one of its own earlier nodes.
__device__ void tours_block(const TourArgs &a, int t, const BlockGroup &g, TourShared &sh) {
    constexpr int I = kChunkItems;
    const int64_t base = a.tree_off[t];
    const int count = static_cast<int>(a.tree_off[t + 1] - base);
    if (g.rank == 0) a.root_depth[t] = 0;
    const int32_t *par = a.parent + base;
    const int32_t *tax = a.taxon + base;
    volatile int32_t *stamp = sh.stamp;
    const int l0 = g.rank * I;  // first chunk slot of this thread
    for (int c0 = 0; c0 < count; c0 += kTourChunk) {
        int p[I];
        double own[I];
        bool pending[I], any = false;
        auto resolve = [&](int l, double v, int d, int s) {
            sh.val[l] = v;
            sh.depth[l] = d;
            stamp[l] = s;
            a.val_s[base + c0 + l] = v;
            a.depth_s[base + c0 + l] = d;
        };
#pragma unroll
        for (int i = 0; i < I; ++i) {
            const int k = c0 + l0 + i;
            const bool internal = k < count && tax[k] < 0;
            pending[i] = false;
            p[i] = 0;
            own[i] = 0.0;
            if (!internal) continue;
            if (k == 0) {  // the value handed to the root's children is 0 (scs.py:577)
                resolve(l0 + i, 0.0, 0, 1);
                continue;
            }
            p[i] = par[k];
            own[i] = own_value(a, base + k);
            if (p[i] < c0) {
                resolve(l0 + i, value_below(a.weighting, a.val_s[base + p[i]], own[i]), a.depth_s[base + p[i]] + 1, 1);
            } else {
                stamp[l0 + i] = 0;
                pending[i] = true;
                any = true;
            }
        }
        for (int round = 1; __syncthreads_or(any); ++round) {
            any = false;
#pragma unroll
            for (int i = 0; i < I; ++i) {
                if (!pending[i]) continue;
                const int q = p[i] - c0;
                const int s = stamp[q];
                if (s > 0 && (s <= round || (q >= l0 && q < l0 + i))) {
                    resolve(l0 + i, value_below(a.weighting, sh.val[q], own[i]), sh.depth[q] + 1, round + 1);
                    pending[i] = false;
                } else {
                    any = true;
                }
            }
        }
    }
    const int64_t o = a.leaf_off[t];
    int tip_base = 0;
    for (int c0 = 0; c0 < count; c0 += kTourChunk) {
        bool tip[I];
        int mine = 0;
#pragma unroll
        for (int i = 0; i < I; ++i) {
            const int k = c0 + l0 + i;
            tip[i] = k < count && tax[k] >= 0;
            mine += tip[i];
        }
        int total;
        int64_t pos = o + tip_base + g.excl_scan(mine, total);
#pragma unroll
        for (int i = 0; i < I; ++i)
            if (tip[i]) write_tip(a, base, count, c0 + l0 + i, pos++);
        tip_base += total;
    }
}

__global__ void __launch_bounds__(kBlock) df_tours(int T, TourArgs a) {
    __shared__ int warp_sum[kWarps];
    __shared__ TourShared sh;
    const BlockGroup block{static_cast<int>(threadIdx.x), warp_sum};
    const int lane = threadIdx.x & 31;
    for_each_item(
        T, [&](int t) { return a.tree_off[t + 1] - a.tree_off[t] > kCtaNodes; },
        [&](int t) { tours_block(a, t, block, sh); }, [&](int t) { tours_warp(a, t, lane); });
}

// ---- restriction ---------------------------------------------------------------------------------------------------
struct RestrictPlan {
    const int32_t *job_tree_begin;  // [J + 1]
    const int32_t *job_parts;       // [J]
    const int32_t *job_part_base;   // [J]
    const int32_t *job_cell_base;   // [J + 1]: cells of job j = parts x trees, cell = base + part * trees + tree
    const int32_t *part_newjob;     // [parts]
    const int32_t *owner;           // [taxa]
    int J;
};

// tips of every tree counted per part of the tree's job; a thread per node, one atomic per cell and warp
__global__ void __launch_bounds__(kBlock)
df_count(int64_t M, int64_t T, const int64_t *__restrict__ tree_off, const int32_t *__restrict__ taxon,
         const int32_t *__restrict__ tree_job, RestrictPlan plan, int32_t *__restrict__ hist) {
    const int64_t g = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
    int cell = -1;
    const int x = g < M ? taxon[g] : -1;
    if (x >= 0) {
        int64_t lo = 0, hi = T;  // the tree of node g: last tree starting at or before it
        while (hi - lo > 1) {
            const int64_t mid = (lo + hi) >> 1;
            if (tree_off[mid] <= g) lo = mid; else hi = mid;
        }
        const int64_t t = lo;
        const int j = tree_job[t];
        const int parts = plan.job_parts[j];
        const int part = plan.owner[x] - plan.job_part_base[j];
        // a tree of fewer than 3 nodes has fewer than two tips
        if (parts > 0 && tree_off[t + 1] - tree_off[t] >= 3 && part >= 0 && part < parts) {
            const int tb = plan.job_tree_begin[j];
            cell = plan.job_cell_base[j] + part * (plan.job_tree_begin[j + 1] - tb) + static_cast<int>(t - tb);
        }
    }
    const unsigned peers = __match_any_sync(kFull, cell);
    if (cell >= 0 && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&hist[cell], __popc(peers));
}

__global__ void df_flag_cells(int cells, const int32_t *__restrict__ hist, int32_t *__restrict__ flag) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < cells) flag[c] = hist[c] >= 2;  // scs.py:447-448: a tree with fewer than two tips of the part is dropped
}

// one entry per (tree, part) pair that yields a restricted tree, in cell order = by new job, trees in source order.
// The per-pair arrays have an entry per cell: those past the pair count are zeroed, so that scans over all cells end
// at the pairs' totals.
__global__ void df_make_pairs(int cells, const int32_t *__restrict__ hist, const int32_t *__restrict__ pair_index,
                              const int64_t *__restrict__ tree_off, RestrictPlan plan, int32_t *__restrict__ pair_count,
                              int32_t *__restrict__ pair_tree, int32_t *__restrict__ pair_part, int32_t *__restrict__ pair_tips,
                              int32_t *__restrict__ pair_need, int32_t *__restrict__ pair_nodes) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cells) return;
    const int pairs = pair_index[cells];
    if (c == 0) *pair_count = pairs;
    if (c >= pairs) pair_tips[c] = pair_need[c] = pair_nodes[c] = 0;
    if (hist[c] < 2) return;
    int lo = 0, hi = plan.J;  // last job with cell_base <= c (jobs without cells share a base with their successor)
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (plan.job_cell_base[mid] <= c) lo = mid; else hi = mid;
    }
    const int j = lo;
    const int trees = plan.job_tree_begin[j + 1] - plan.job_tree_begin[j];
    const int within = c - plan.job_cell_base[j];
    const int part = within / trees, tl = within - part * trees;
    const int t = plan.job_tree_begin[j] + tl;
    const int p = pair_index[c];
    pair_tree[p] = t;
    pair_part[p] = plan.job_part_base[j] + part;
    pair_tips[p] = hist[c];
    pair_need[p] = static_cast<int32_t>(tree_off[t + 1] - tree_off[t]) + 1;
}

// A pair is walked by a CTA when its tree has more than kCtaNodes nodes (need = nodes + 1).
struct PairList {
    const int32_t *count, *tree, *part, *tips, *need, *scratch_off;
};

__device__ __forceinline__ bool large_pair(const PairList &pl, int p) { return pl.need[p] > kCtaNodes + 1; }

// kept / retained prefix sums of one (tree, part) pair
template <class G>
__device__ void mark_pair(const G &g, int p, const PairList &pl, const int64_t *__restrict__ tree_off,
                          const int32_t *__restrict__ parent, const int32_t *__restrict__ size,
                          const int32_t *__restrict__ taxon, const int32_t *__restrict__ owner, int32_t *P_all,
                          int32_t *R_all, uint8_t *U_all, int32_t *__restrict__ pair_nodes) {
    constexpr int I = G::kItems, kChunk = G::kSize * G::kItems;
    const int t = pl.tree[p], part = pl.part[p];
    const int64_t base = tree_off[t];
    const int count = static_cast<int>(tree_off[t + 1] - base);
    const int32_t *par = parent + base;
    const int32_t *sz = size + base;
    const int32_t *tax = taxon + base;
    int32_t *P = P_all + pl.scratch_off[p];
    int32_t *R = R_all + pl.scratch_off[p];
    uint8_t *U = U_all + pl.scratch_off[p];
    int carry = 0;
    for (int c0 = 0; c0 < count; c0 += kChunk) {
        const int k0 = c0 + g.rank * I;
        int kept[I], mine = 0;
#pragma unroll
        for (int i = 0; i < I; ++i) {
            const int k = k0 + i;
            kept[i] = 0;
            if (k < count) {
                const int x = tax[k];
                kept[i] = x >= 0 && owner[x] == part;
                U[k] = 0;
            }
            mine += kept[i];
        }
        int total;
        int run = carry + g.excl_scan(mine, total);
#pragma unroll
        for (int i = 0; i < I; ++i) {
            if (k0 + i < count) P[k0 + i] = run;
            run += kept[i];
        }
        carry += total;
    }
    if (g.rank == 0) P[count] = carry;
    g.sync();
    for (int k = 1 + g.rank; k < count; k += G::kSize) {
        const int cnt = P[k + sz[k]] - P[k];
        if (cnt > 0) {
            const int up = par[k];
            if (cnt == P[up + sz[up]] - P[up]) U[up] = 1;  // the parent has all its kept tips below this child
        }
    }
    g.sync();
    carry = 0;
    for (int c0 = 0; c0 < count; c0 += kChunk) {
        const int k0 = c0 + g.rank * I;
        int retained[I], mine = 0;
#pragma unroll
        for (int i = 0; i < I; ++i) {
            const int k = k0 + i;
            retained[i] = 0;
            if (k < count) {
                const int cnt = P[k + sz[k]] - P[k];
                retained[i] = cnt > 0 && (tax[k] >= 0 || !U[k]);
            }
            mine += retained[i];
        }
        int total;
        int run = carry + g.excl_scan(mine, total);
#pragma unroll
        for (int i = 0; i < I; ++i) {
            if (k0 + i < count) R[k0 + i] = run;
            run += retained[i];
        }
        carry += total;
    }
    if (g.rank == 0) {
        R[count] = carry;
        pair_nodes[p] = carry;
    }
    g.sync();  // a CTA's next pair reuses the scan's shared memory
}

__global__ void __launch_bounds__(kBlock)
df_mark(PairList pl, const int64_t *__restrict__ tree_off, const int32_t *__restrict__ parent,
        const int32_t *__restrict__ size, const int32_t *__restrict__ taxon, const int32_t *__restrict__ owner,
        int32_t *P_all, int32_t *R_all, uint8_t *U_all, int32_t *__restrict__ pair_nodes) {
    __shared__ int warp_sum[kWarps];
    const BlockGroup block{static_cast<int>(threadIdx.x), warp_sum};
    const WarpGroup warp{static_cast<int>(threadIdx.x & 31)};
    for_each_item(
        *pl.count, [&](int p) { return large_pair(pl, p); },
        [&](int p) { mark_pair(block, p, pl, tree_off, parent, size, taxon, owner, P_all, R_all, U_all, pair_nodes); },
        [&](int p) { mark_pair(warp, p, pl, tree_off, parent, size, taxon, owner, P_all, R_all, U_all, pair_nodes); });
}

struct WriteOut {
    int32_t *parent, *size, *taxon;
    double *length, *support, *weight;
    int64_t *tree_off, *leaf_off;
    int32_t *tree_job;
    uint8_t *present;
    int32_t *job_trees;
    unsigned long long *job_visits;
};

// the restricted tree of one pair written into the new forest
template <class G>
__device__ void write_pair(const G &g, int p, int pairs, const PairList &pl, const int32_t *__restrict__ node_off32,
                           const int32_t *__restrict__ leaf_off32, const int32_t *__restrict__ part_newjob,
                           const int64_t *__restrict__ tree_off, const int32_t *__restrict__ parent,
                           const int32_t *__restrict__ size, const int32_t *__restrict__ taxon,
                           const double *__restrict__ length, const double *__restrict__ support,
                           const double *__restrict__ weight, const int32_t *__restrict__ R_all, const WriteOut &o) {
    const int t = pl.tree[p];
    const int64_t base = tree_off[t];
    const int count = static_cast<int>(tree_off[t + 1] - base);
    const int32_t *par = parent + base;
    const int32_t *sz = size + base;
    const int32_t *tax = taxon + base;
    const int32_t *R = R_all + pl.scratch_off[p];
    const int64_t ob = node_off32[p];
    const double nan_v = __longlong_as_double(0x7ff8000000000000ll);
    for (int k = g.rank; k < count; k += G::kSize) {
        const int q = R[k];
        if (R[k + 1] == q) continue;  // not retained
        int up = -1;
        double acc = nan_v;
        if (q > 0) {
            // merged unary ancestors, bottom-up: length(node) + length(child); NaN (missing) propagates like None
            up = par[k];
            if (length) acc = length[base + k];
            while (R[up + 1] == R[up]) {
                if (length) acc = __dadd_rn(length[base + up], acc);
                up = par[up];
            }
            up = R[up];
        }
        // q == 0: the first retained node in pre-order is the new root; its own length is dropped
        o.parent[ob + q] = up;
        o.size[ob + q] = R[k + sz[k]] - q;
        o.taxon[ob + q] = tax[k];
        if (o.length) o.length[ob + q] = acc;
        if (o.support) o.support[ob + q] = support[base + k];
        if (tax[k] >= 0) o.present[tax[k]] = 1;  // racing writers all store 1
    }
    if (g.rank == 0) {
        const int job = part_newjob[pl.part[p]];
        o.weight[p] = weight[t];
        o.tree_job[p] = job;
        o.tree_off[p] = ob;
        o.leaf_off[p] = leaf_off32[p];
        if (p == pairs - 1) {
            o.tree_off[pairs] = node_off32[pairs];
            o.leaf_off[pairs] = leaf_off32[pairs];
        }
        if (job >= 0) {  // always: taxa of parts without a job have owner -1 and never make a pair
            atomicAdd(&o.job_trees[job], 1);
            const unsigned long long k = static_cast<unsigned long long>(pl.tips[p]);
            atomicAdd(&o.job_visits[job], k * (k - 1ull));
        }
    }
}

__global__ void __launch_bounds__(kBlock)
df_write(PairList pl, const int32_t *__restrict__ node_off32, const int32_t *__restrict__ leaf_off32,
         const int32_t *__restrict__ part_newjob, const int64_t *__restrict__ tree_off, const int32_t *__restrict__ parent,
         const int32_t *__restrict__ size, const int32_t *__restrict__ taxon, const double *__restrict__ length,
         const double *__restrict__ support, const double *__restrict__ weight, const int32_t *__restrict__ R_all, WriteOut o) {
    const int pairs = *pl.count;
    const BlockGroup block{static_cast<int>(threadIdx.x), nullptr};
    const WarpGroup warp{static_cast<int>(threadIdx.x & 31)};
    for_each_item(
        pairs, [&](int p) { return large_pair(pl, p); },
        [&](int p) {
            write_pair(block, p, pairs, pl, node_off32, leaf_off32, part_newjob, tree_off, parent, size, taxon, length,
                       support, weight, R_all, o);
        },
        [&](int p) {
            write_pair(warp, p, pairs, pl, node_off32, leaf_off32, part_newjob, tree_off, parent, size, taxon, length,
                       support, weight, R_all, o);
        });
}

__global__ void df_job_info(int jobs, const int32_t *__restrict__ job_trees, const int32_t *__restrict__ job_tree_begin,
                            const int32_t *__restrict__ node_off32, const int32_t *__restrict__ leaf_off32,
                            const unsigned long long *__restrict__ job_visits, DevJobInfo *__restrict__ info) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= jobs) return;
    DevJobInfo out;
    out.trees = job_trees[j];
    out.tree_begin = job_tree_begin[j];
    out.leaf_begin = leaf_off32[out.tree_begin];
    out.node_begin = node_off32[out.tree_begin];
    out.first_tree_nodes = out.trees > 0 ? node_off32[out.tree_begin + 1] - node_off32[out.tree_begin] : 0;
    out.pair_visits = static_cast<int64_t>(job_visits[j]);
    info[j] = out;
}

struct FetchItem {
    int64_t src, dst, count;
};

__global__ void df_fetch(int items, const FetchItem *__restrict__ item, const int32_t *__restrict__ parent,
                         const int32_t *__restrict__ taxon, int32_t *__restrict__ o_parent, int32_t *__restrict__ o_taxon) {
    const int i = blockIdx.x;
    if (i >= items) return;
    const FetchItem it = item[i];
    for (int64_t k = threadIdx.x; k < it.count; k += blockDim.x) {
        o_parent[it.dst + k] = parent[it.src + k];
        o_taxon[it.dst + k] = taxon[it.src + k];
    }
}

template <typename T>
T *carve(unsigned char *&cursor, size_t count) {
    T *out = reinterpret_cast<T *>(cursor);
    cursor += (count * sizeof(T) + 255) & ~static_cast<size_t>(255);
    return out;
}

}  // namespace

int devforest_upload(scs_ctx *ctx, const scs_forest *host, int weighting, DevForest *out, bool cooperative) {
    if (!host || !out) return fail(ctx, SCS_ERR_INVALID, "devforest_upload: bad argument");
    const int64_t T = host->num_trees(), M = host->node_offsets.back();
    if (M >= (1ll << 31)) return fail(ctx, SCS_ERR_INVALID, "device forest: more than 2^31 tree nodes");
    out->trees = T;
    out->nodes = M;
    out->leaves = host->leaf_offsets.back();
    out->has_length = weighting == 1;
    out->has_support = weighting == 3;
    int rc;
    const size_t nT = static_cast<size_t>(T), nM = static_cast<size_t>(M);
    if ((rc = grow(ctx, out->tree_off, (nT + 1) * sizeof(int64_t)))) return rc;
    if ((rc = grow(ctx, out->leaf_off, (nT + 1) * sizeof(int64_t)))) return rc;
    if ((rc = grow(ctx, out->parent, nM * sizeof(int32_t)))) return rc;
    if ((rc = grow(ctx, out->size, nM * sizeof(int32_t)))) return rc;
    if ((rc = grow(ctx, out->taxon, nM * sizeof(int32_t)))) return rc;
    if ((rc = grow(ctx, out->weight, nT * sizeof(double)))) return rc;
    if ((rc = grow(ctx, out->tree_job, nT * sizeof(int32_t)))) return rc;
    if (out->has_length && (rc = grow(ctx, out->length, nM * sizeof(double)))) return rc;
    if (out->has_support && (rc = grow(ctx, out->support, nM * sizeof(double)))) return rc;

    // the per-node arrays, and where each starts in a rank's staging area (the W block of its exchange window)
    struct NodeArray {
        GrowBuf *dst;
        const void *src;  // null: the subtree sizes, computed below
        size_t elem, stage_off;
    };
    std::vector<NodeArray> arrays = {{&out->parent, host->parent.data(), sizeof(int32_t), 0},
                                     {&out->size, nullptr, sizeof(int32_t), 0},
                                     {&out->taxon, host->taxon.data(), sizeof(int32_t), 0}};
    if (out->has_length) arrays.push_back({&out->length, host->length.data(), sizeof(double), 0});
    if (out->has_support) arrays.push_back({&out->support, host->support.data(), sizeof(double), 0});
    size_t stage_bytes = 0;
    for (NodeArray &a : arrays) {
        a.stage_off = stage_bytes;
        stage_bytes += (nM * a.elem + 255) & ~static_cast<size_t>(255);
    }
    ShardState &sh = ctx->shard;
    // worth it from a few million nodes (below that the barriers cost more than the link saves); tests lower the bar
    const char *min_nodes_env = std::getenv("SCS_SHARED_UPLOAD_MIN_NODES");
    const size_t min_nodes = min_nodes_env ? static_cast<size_t>(std::atoll(min_nodes_env)) : (1u << 22);
    const bool share = cooperative && sh.connected && sh.world > 1 && nM > min_nodes &&
                       sh.layout.total > sh.layout.W && stage_bytes <= sh.layout.total - sh.layout.W;
    const int G = share ? sh.world : 1, me = share ? sh.rank : 0;
    auto slice_begin = [&](int p) { return static_cast<int64_t>(M * static_cast<__int128>(p) / G); };
    const int64_t lo = slice_begin(me), hi = slice_begin(me + 1);

    // subtree sizes (pre-order: the nodes of a subtree are a contiguous run) of the trees that overlap this rank's
    // slice, per tree, over the host threads
    const int64_t *offs = host->node_offsets.data();
    const int64_t t_lo = hi > lo ? std::upper_bound(offs, offs + T + 1, lo) - offs - 1 : 0;
    const int64_t t_hi = hi > lo ? std::lower_bound(offs, offs + T + 1, hi) - offs : 0;
    const int64_t size_base = T > 0 && hi > lo ? offs[t_lo] : 0;
    std::vector<int32_t> size(static_cast<size_t>(hi > lo ? offs[t_hi] - size_base : 1));
#pragma omp parallel for schedule(dynamic, 16) num_threads(scs_host_threads()) if (M > (1 << 15))
    for (int64_t t = t_lo; t < t_hi; ++t) {
        const int64_t base = offs[t], count = offs[t + 1] - base;
        int32_t *sz = size.data() + (base - size_base);
        for (int64_t k = 0; k < count; ++k) sz[k] = 1;
        for (int64_t k = count - 1; k >= 1; --k) sz[host->parent[base + k]] += sz[k];
    }

    // Pageable memory goes to the device through two pinned chunks: the host threads fill one while the other is on
    // the wire (a plain cudaMemcpy from pageable memory stages serially through the driver at a fraction of the
    // link's rate: 0.26 s for the 0.8 GB of the 50 000-taxon workload).
    constexpr size_t kChunk = 32u << 20;
    const bool staged = nM * sizeof(double) > (8u << 20);
    unsigned char *pin = nullptr;
    cudaEvent_t sent[2] = {nullptr, nullptr};
    if (staged) {
        void *pin_v;
        if ((rc = reserve_pinned(ctx, 2 * kChunk, &pin_v))) return rc;
        pin = static_cast<unsigned char *>(pin_v);
        for (cudaEvent_t &e : sent) SCS_CUDA(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    int turn = 0;
    const int copy_threads = scs_host_threads() > 0 ? scs_host_threads() : 1;
    auto put = [&](void *dst, const void *src, size_t bytes) -> int {
        if (bytes == 0) return SCS_OK;
        ctx->h2d_bytes += static_cast<int64_t>(bytes);
        if (!staged || bytes < (1u << 20)) {
            SCS_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
            return SCS_OK;
        }
        for (size_t at = 0; at < bytes; at += kChunk, turn ^= 1) {
            const size_t len = bytes - at < kChunk ? bytes - at : kChunk;
            unsigned char *stage = pin + static_cast<size_t>(turn) * kChunk;
            SCS_CUDA(ctx, cudaEventSynchronize(sent[turn]));  // the chunk's previous copy has left it
            const long long pieces = static_cast<long long>((len + (1u << 20) - 1) >> 20);
#pragma omp parallel for schedule(static) num_threads(copy_threads)
            for (long long p = 0; p < pieces; ++p) {
                const size_t o = static_cast<size_t>(p) << 20;
                std::memcpy(stage + o, static_cast<const unsigned char *>(src) + at + o, len - o < (1u << 20) ? len - o : (1u << 20));
            }
            SCS_CUDA(ctx, cudaMemcpyAsync(static_cast<unsigned char *>(dst) + at, stage, len, cudaMemcpyHostToDevice, ctx->stream));
            SCS_CUDA(ctx, cudaEventRecord(sent[turn], ctx->stream));
        }
        return SCS_OK;
    };
    if ((rc = put(out->tree_off.ptr, host->node_offsets.data(), (nT + 1) * sizeof(int64_t)))) return rc;
    if ((rc = put(out->leaf_off.ptr, host->leaf_offsets.data(), (nT + 1) * sizeof(int64_t)))) return rc;
    if ((rc = put(out->weight.ptr, host->weight.data(), nT * sizeof(double)))) return rc;
    SCS_CUDA(ctx, cudaMemsetAsync(out->tree_job.ptr, 0, nT * sizeof(int32_t), ctx->stream));
    const size_t n_mine = static_cast<size_t>(hi - lo);
    auto source_of = [&](const NodeArray &a) -> const unsigned char * {
        if (a.src) return static_cast<const unsigned char *>(a.src) + static_cast<size_t>(lo) * a.elem;
        return reinterpret_cast<const unsigned char *>(size.data() + (lo - size_base));
    };
    if (!share) {
        for (const NodeArray &a : arrays)
            if ((rc = put(a.dst->ptr, source_of(a), n_mine * a.elem))) return rc;
    } else {
        // nobody may still be reading this rank's W block (the last shared node of a previous build)
        if ((rc = shard_barrier(ctx))) return rc;
        unsigned char *stage = sh.window + sh.layout.W;
        for (const NodeArray &a : arrays)
            if ((rc = put(stage + a.stage_off + static_cast<size_t>(lo) * a.elem, source_of(a), n_mine * a.elem))) return rc;
        if ((rc = shard_barrier(ctx))) return rc;  // every rank's slice is in its window
        for (int step = 0; step < G; ++step) {
            const int p = (me + step) % G;  // staggered so that the ranks do not all read one peer
            const size_t b = static_cast<size_t>(slice_begin(p)), e = static_cast<size_t>(slice_begin(p + 1));
            for (const NodeArray &a : arrays) {
                if (e == b) continue;
                SCS_CUDA(ctx, cudaMemcpyAsync(static_cast<unsigned char *>(a.dst->ptr) + b * a.elem,
                                              sh.peer[p] + sh.layout.W + a.stage_off + b * a.elem, (e - b) * a.elem,
                                              cudaMemcpyDeviceToDevice, ctx->stream));
            }
        }
        if ((rc = shard_barrier(ctx))) return rc;  // the windows are free again
    }
    // `size` is a local: the copies above must have read it before it goes away
    SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (cudaEvent_t e : sent)
        if (e) cudaEventDestroy(e);
    if (share) {
        // a peer that timed out in one of the barriers leaves its mark in the window header
        unsigned int error = 0;
        SCS_CUDA(ctx, cudaMemcpy(&error, sh.window + offsetof(ShardHeader, error), sizeof(error), cudaMemcpyDeviceToHost));
        if (error) return fail(ctx, SCS_ERR_PEER, "device forest: a wait for a peer GPU timed out");
    }
    return SCS_OK;
}

// blocks of a launch over `items` trees or pairs (for_each_item): a block per item up to a full load of the GPU
static int item_blocks(const scs_ctx *ctx, int64_t items) {
    const int64_t full = static_cast<int64_t>(ctx->sm_count) * (2048 / kBlock);
    return static_cast<int>(std::max<int64_t>(1, std::min(items, full)));
}

int devforest_tours(scs_ctx *ctx, const DevForest &f, int weighting, const int32_t *taxon_vertex_dev, DevTours *tours,
                    int32_t *flags_dev) {
    int rc;
    const size_t nL = static_cast<size_t>(f.leaves), nT = static_cast<size_t>(f.trees), nM = static_cast<size_t>(f.nodes);
    if ((rc = grow(ctx, tours->leaf_taxon, (nL + 1) * sizeof(int32_t)))) return rc;
    if ((rc = grow(ctx, tours->adj_depth, (nL + 1) * sizeof(int32_t)))) return rc;
    if ((rc = grow(ctx, tours->adj_val, (nL + 1) * sizeof(double)))) return rc;
    if ((rc = grow(ctx, tours->root_depth, (nT + 1) * sizeof(int32_t)))) return rc;
    if ((rc = grow(ctx, tours->depth_s, (nM + 1) * sizeof(int32_t)))) return rc;
    if ((rc = grow(ctx, tours->val_s, (nM + 1) * sizeof(double)))) return rc;
    if (f.trees == 0) return SCS_OK;
    TourArgs a;
    a.tree_off = f.tree_off.as<int64_t>();
    a.leaf_off = f.leaf_off.as<int64_t>();
    a.parent = f.parent.as<int32_t>();
    a.taxon = f.taxon.as<int32_t>();
    a.length = f.has_length ? f.length.as<double>() : nullptr;
    a.support = f.has_support ? f.support.as<double>() : nullptr;
    a.weighting = weighting;
    a.taxon_vertex = taxon_vertex_dev;
    a.depth_s = tours->depth_s.as<int32_t>();
    a.val_s = tours->val_s.as<double>();
    a.leaf_taxon = tours->leaf_taxon.as<int32_t>();
    a.adj_depth = tours->adj_depth.as<int32_t>();
    a.adj_val = tours->adj_val.as<double>();
    a.root_depth = tours->root_depth.as<int32_t>();
    a.flags = flags_dev;
    df_tours<<<item_blocks(ctx, f.trees), kBlock, 0, ctx->stream>>>(static_cast<int>(f.trees), a);
    SCS_LAUNCHED(ctx, "df_tours");
    return SCS_OK;
}

int devforest_restrict(scs_ctx *ctx, const DevForest &src, int J, const int32_t *job_tree_begin, const int64_t *job_node_begin,
                       const int32_t *job_parts, const int32_t *job_part_base, int num_parts, const int32_t *part_newjob,
                       int new_jobs, const int32_t *owner_host, int num_taxa, DevForest *dst, DevJobInfo *info,
                       uint8_t *present_host) {
    if (J <= 0 || !job_tree_begin || !job_node_begin || !job_parts || !job_part_base || !part_newjob || !owner_host || !dst ||
        !info || !present_host)
        return fail(ctx, SCS_ERR_INVALID, "devforest_restrict: bad argument");
    // cells: one per (part, tree) of every job that was split.  A pair's scratch is its tree's nodes + 1, so the
    // scratch of job j's pairs is at most parts x (nodes + trees) of the job.
    std::vector<int32_t> cell_base(static_cast<size_t>(J) + 1, 0);
    int64_t cells = 0, scratch_bound = 0;
    for (int j = 0; j < J; ++j) {
        cell_base[j] = static_cast<int32_t>(cells);
        const int64_t trees = job_tree_begin[j + 1] - job_tree_begin[j];
        cells += static_cast<int64_t>(job_parts[j]) * trees;
        scratch_bound += static_cast<int64_t>(job_parts[j]) * (job_node_begin[j + 1] - job_node_begin[j] + trees);
        if (cells >= (1ll << 31) - 8) return fail(ctx, SCS_ERR_INVALID, "device forest: too many (tree, part) cells");
    }
    cell_base[J] = static_cast<int32_t>(cells);
    dst->has_length = src.has_length;
    dst->has_support = src.has_support;
    const size_t nJ = static_cast<size_t>(J), nP = static_cast<size_t>(num_parts > 0 ? num_parts : 1), nX = static_cast<size_t>(num_taxa),
                 nC = static_cast<size_t>(cells), nN = static_cast<size_t>(new_jobs > 0 ? new_jobs : 1);
    std::memset(present_host, 0, nX);
    if (cells == 0 || new_jobs == 0) {
        dst->trees = dst->nodes = dst->leaves = 0;
        for (int j = 0; j < new_jobs; ++j) info[j] = DevJobInfo{0, 0, 0, 0, 0, 0};
        return SCS_OK;
    }
    int rc;
    // ---- plan tables + owner: one pinned staging block, one copy -----------------------------------------------------
    const size_t plan_bytes = (4 * (nJ + 1) + nP + nX) * sizeof(int32_t) + 2048;
    void *pin_v;
    if ((rc = reserve_pinned(ctx, plan_bytes + nX + sizeof(DevJobInfo) * nN + 4096, &pin_v))) return rc;
    unsigned char *pin = static_cast<unsigned char *>(pin_v);
    unsigned char *plan_dev_raw;
    if ((rc = reserve_as(ctx, SLOT_MED_STAGE, plan_bytes, &plan_dev_raw))) return rc;
    size_t at = 0;
    auto stage = [&](const int32_t *srcp, size_t count) {
        const size_t here = at;
        std::memcpy(pin + here, srcp, count * sizeof(int32_t));
        at += (count * sizeof(int32_t) + 255) & ~static_cast<size_t>(255);
        return here;
    };
    const size_t o_tb = stage(job_tree_begin, nJ + 1), o_parts = stage(job_parts, nJ), o_pbase = stage(job_part_base, nJ),
                 o_cbase = stage(cell_base.data(), nJ + 1), o_newjob = stage(part_newjob, nP), o_owner = stage(owner_host, nX);
    SCS_CUDA(ctx, cudaMemcpyAsync(plan_dev_raw, pin, at, cudaMemcpyHostToDevice, ctx->stream));
    ctx->h2d_bytes += static_cast<int64_t>(at);
    RestrictPlan plan;
    plan.job_tree_begin = reinterpret_cast<const int32_t *>(plan_dev_raw + o_tb);
    plan.job_parts = reinterpret_cast<const int32_t *>(plan_dev_raw + o_parts);
    plan.job_part_base = reinterpret_cast<const int32_t *>(plan_dev_raw + o_pbase);
    plan.job_cell_base = reinterpret_cast<const int32_t *>(plan_dev_raw + o_cbase);
    plan.part_newjob = reinterpret_cast<const int32_t *>(plan_dev_raw + o_newjob);
    plan.owner = reinterpret_cast<const int32_t *>(plan_dev_raw + o_owner);
    plan.J = J;

    // ---- workspaces: every per-pair array has an entry per cell (cells bound the pairs), the jobs' counters -----------
    unsigned char *wa;
    if ((rc = reserve_as(ctx, SLOT_MED_STATE, 3 * ((nC + 2) * sizeof(int32_t) + 256) + 1024, &wa))) return rc;
    int32_t *hist = carve<int32_t>(wa, nC + 1);
    int32_t *flag = carve<int32_t>(wa, nC + 1);
    int32_t *pair_index = carve<int32_t>(wa, nC + 2);
    unsigned char *wb;
    if ((rc = reserve_as(ctx, SLOT_MED_VEC, 9 * ((nC + 2) * sizeof(int32_t) + 256) + 2 * (nN + 2) * sizeof(int32_t) +
                                               (nN + 1) * sizeof(unsigned long long) + nX + 4096, &wb)))
        return rc;
    int32_t *pair_tree = carve<int32_t>(wb, nC + 1);
    int32_t *pair_part = carve<int32_t>(wb, nC + 1);
    int32_t *pair_tips = carve<int32_t>(wb, nC + 1);
    int32_t *pair_need = carve<int32_t>(wb, nC + 1);
    int32_t *scratch_off = carve<int32_t>(wb, nC + 2);
    int32_t *pair_nodes = carve<int32_t>(wb, nC + 1);
    int32_t *node_off32 = carve<int32_t>(wb, nC + 2);
    int32_t *leaf_off32 = carve<int32_t>(wb, nC + 2);
    int32_t *pair_count_dev = carve<int32_t>(wb, 64);
    unsigned char *counters = wb;  // job_trees .. present: zeroed in one piece
    int32_t *job_trees = carve<int32_t>(wb, nN + 1);
    int32_t *job_tree_begin_new = carve<int32_t>(wb, nN + 2);
    unsigned long long *job_visits = carve<unsigned long long>(wb, nN + 1);
    uint8_t *present = carve<uint8_t>(wb, nX + 1);
    SCS_CUDA(ctx, cudaMemsetAsync(hist, 0, (nC + 1) * sizeof(int32_t), ctx->stream));
    SCS_CUDA(ctx, cudaMemsetAsync(counters, 0, static_cast<size_t>(wb - counters), ctx->stream));

    // ---- which (tree, part) pairs exist ---------------------------------------------------------------------------------
    const int64_t T = src.trees;
    df_count<<<ceil_div(src.nodes, kBlock), kBlock, 0, ctx->stream>>>(src.nodes, T, src.tree_off.as<int64_t>(),
                                                                     src.taxon.as<int32_t>(), src.tree_job.as<int32_t>(),
                                                                     plan, hist);
    SCS_LAUNCHED(ctx, "df_count");
    const int ncells = static_cast<int>(cells);
    df_flag_cells<<<ceil_div(ncells, 256), 256, 0, ctx->stream>>>(ncells, hist, flag);
    SCS_LAUNCHED(ctx, "df_flag_cells");
    if ((rc = exclusive_scan(ctx, ncells, flag, pair_index))) return rc;
    df_make_pairs<<<ceil_div(ncells, 256), 256, 0, ctx->stream>>>(ncells, hist, pair_index, src.tree_off.as<int64_t>(), plan,
                                                                 pair_count_dev, pair_tree, pair_part, pair_tips, pair_need,
                                                                 pair_nodes);
    SCS_LAUNCHED(ctx, "df_make_pairs");
    if ((rc = exclusive_scan(ctx, ncells, pair_need, scratch_off))) return rc;
    // P | R | U per (pair, node), sized by the bound; a split into many parts can make the bound far larger than what
    // the pairs use: past the cap the exact size is read back first
    int32_t *pin_counts = reinterpret_cast<int32_t *>(pin + plan_bytes);
    size_t scratch_entries = static_cast<size_t>(scratch_bound);
    const int64_t scratch_cap = std::min<int64_t>(std::max<int64_t>(4 * (src.nodes + src.trees), 1ll << 22), (1ll << 31) - 1024);
    if (scratch_bound > scratch_cap) {
        SCS_CUDA(ctx, cudaMemcpyAsync(pin_counts + 1, scratch_off + ncells, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        scratch_entries = static_cast<size_t>(pin_counts[1]);
    }
    unsigned char *wc;
    if ((rc = reserve_as(ctx, SLOT_BASIS, 2 * (scratch_entries * sizeof(int32_t) + 256) + scratch_entries + 1024, &wc))) return rc;
    int32_t *P_all = carve<int32_t>(wc, scratch_entries);
    int32_t *R_all = carve<int32_t>(wc, scratch_entries);
    uint8_t *U_all = carve<uint8_t>(wc, scratch_entries);
    const PairList pl{pair_count_dev, pair_tree, pair_part, pair_tips, pair_need, scratch_off};
    const int pair_blocks = item_blocks(ctx, cells);
    df_mark<<<pair_blocks, kBlock, 0, ctx->stream>>>(pl, src.tree_off.as<int64_t>(), src.parent.as<int32_t>(),
                                                    src.size.as<int32_t>(), src.taxon.as<int32_t>(), plan.owner, P_all, R_all,
                                                    U_all, pair_nodes);
    SCS_LAUNCHED(ctx, "df_mark");
    if ((rc = exclusive_scan(ctx, ncells, pair_nodes, node_off32))) return rc;
    if ((rc = exclusive_scan(ctx, ncells, pair_tips, leaf_off32))) return rc;

    // ---- the new forest: at most 2 nodes per kept tip (restricted trees branch everywhere) ------------------------------
    const size_t cap_nodes = 2 * static_cast<size_t>(src.leaves) + 16;
    if ((rc = grow(ctx, dst->tree_off, (nC + 1) * sizeof(int64_t)))) return rc;
    if ((rc = grow(ctx, dst->leaf_off, (nC + 1) * sizeof(int64_t)))) return rc;
    if ((rc = grow(ctx, dst->parent, cap_nodes * sizeof(int32_t)))) return rc;
    if ((rc = grow(ctx, dst->size, cap_nodes * sizeof(int32_t)))) return rc;
    if ((rc = grow(ctx, dst->taxon, cap_nodes * sizeof(int32_t)))) return rc;
    if ((rc = grow(ctx, dst->weight, nC * sizeof(double)))) return rc;
    if ((rc = grow(ctx, dst->tree_job, nC * sizeof(int32_t)))) return rc;
    if (dst->has_length && (rc = grow(ctx, dst->length, cap_nodes * sizeof(double)))) return rc;
    if (dst->has_support && (rc = grow(ctx, dst->support, cap_nodes * sizeof(double)))) return rc;
    WriteOut out;
    out.parent = dst->parent.as<int32_t>();
    out.size = dst->size.as<int32_t>();
    out.taxon = dst->taxon.as<int32_t>();
    out.length = dst->has_length ? dst->length.as<double>() : nullptr;
    out.support = dst->has_support ? dst->support.as<double>() : nullptr;
    out.weight = dst->weight.as<double>();
    out.tree_off = dst->tree_off.as<int64_t>();
    out.leaf_off = dst->leaf_off.as<int64_t>();
    out.tree_job = dst->tree_job.as<int32_t>();
    out.present = present;
    out.job_trees = job_trees;
    out.job_visits = job_visits;
    df_write<<<pair_blocks, kBlock, 0, ctx->stream>>>(
        pl, node_off32, leaf_off32, plan.part_newjob, src.tree_off.as<int64_t>(), src.parent.as<int32_t>(),
        src.size.as<int32_t>(), src.taxon.as<int32_t>(), src.has_length ? src.length.as<double>() : nullptr,
        src.has_support ? src.support.as<double>() : nullptr, src.weight.as<double>(), R_all, out);
    SCS_LAUNCHED(ctx, "df_write");
    if ((rc = exclusive_scan(ctx, new_jobs, job_trees, job_tree_begin_new))) return rc;
    DevJobInfo *info_dev;
    if ((rc = reserve_as(ctx, SLOT_NODE_STATS, nN + 1, &info_dev))) return rc;
    df_job_info<<<ceil_div(new_jobs, 256), 256, 0, ctx->stream>>>(new_jobs, job_trees, job_tree_begin_new, node_off32, leaf_off32,
                                                                 job_visits, info_dev);
    SCS_LAUNCHED(ctx, "df_job_info");
    // ---- the one synchronisation: presence, job info, totals ------------------------------------------------------------
    unsigned char *pin_present = pin + plan_bytes + 256;
    DevJobInfo *pin_info = reinterpret_cast<DevJobInfo *>(pin + plan_bytes + 256 + ((nX + 255) & ~static_cast<size_t>(255)));
    SCS_CUDA(ctx, cudaMemcpyAsync(pin_present, present, nX, cudaMemcpyDeviceToHost, ctx->stream));
    SCS_CUDA(ctx, cudaMemcpyAsync(pin_info, info_dev, sizeof(DevJobInfo) * new_jobs, cudaMemcpyDeviceToHost, ctx->stream));
    SCS_CUDA(ctx, cudaMemcpyAsync(pin_counts, pair_count_dev, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    SCS_CUDA(ctx, cudaMemcpyAsync(pin_counts + 2, node_off32 + ncells, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    SCS_CUDA(ctx, cudaMemcpyAsync(pin_counts + 3, leaf_off32 + ncells, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->d2h_bytes += static_cast<int64_t>(nX + sizeof(DevJobInfo) * new_jobs + 16);
    std::memcpy(present_host, pin_present, nX);
    std::memcpy(info, pin_info, sizeof(DevJobInfo) * new_jobs);
    dst->trees = pin_counts[0];
    dst->nodes = pin_counts[2];
    dst->leaves = pin_counts[3];
    return SCS_OK;
}

int devforest_fetch_trees(scs_ctx *ctx, const DevForest &forest, int count, const int64_t *first_node,
                          const int64_t *tree_nodes, int32_t *parent_out, int32_t *taxon_out) {
    if (count <= 0) return SCS_OK;
    std::vector<FetchItem> items(static_cast<size_t>(count));
    int64_t total = 0;
    for (int i = 0; i < count; ++i) {
        if (first_node[i] < 0 || first_node[i] + tree_nodes[i] > forest.nodes)
            return fail(ctx, SCS_ERR_INVALID, "devforest_fetch_trees: tree outside the forest");
        items[i] = FetchItem{first_node[i], total, tree_nodes[i]};
        total += tree_nodes[i];
    }
    FetchItem *items_dev;
    int32_t *packed;
    int rc;
    if ((rc = reserve_as(ctx, SLOT_MED_ROW_NODE, static_cast<size_t>(count) + 1, &items_dev))) return rc;
    if ((rc = reserve_as(ctx, SLOT_MED_TREE_NODE, 2 * static_cast<size_t>(total) + 8, &packed))) return rc;
    SCS_CUDA(ctx, cudaMemcpyAsync(items_dev, items.data(), sizeof(FetchItem) * count, cudaMemcpyHostToDevice, ctx->stream));
    df_fetch<<<count, 128, 0, ctx->stream>>>(count, items_dev, forest.parent.as<int32_t>(), forest.taxon.as<int32_t>(), packed,
                                            packed + total);
    SCS_LAUNCHED(ctx, "df_fetch");
    SCS_CUDA(ctx, cudaMemcpyAsync(parent_out, packed, sizeof(int32_t) * total, cudaMemcpyDeviceToHost, ctx->stream));
    SCS_CUDA(ctx, cudaMemcpyAsync(taxon_out, packed + total, sizeof(int32_t) * total, cudaMemcpyDeviceToHost, ctx->stream));
    SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // also keeps `items` alive until the copy has read it
    ctx->d2h_bytes += static_cast<int64_t>(2 * sizeof(int32_t) * total);
    return SCS_OK;
}

}  // namespace scs
