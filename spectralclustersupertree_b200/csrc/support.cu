// Source-tree support of the clades of a supertree (scs_supertree_support): for every internal node u of the
// supertree S and every source tree t, the clade A = leaves(u) restricted to the taxa X_t that t and S share is
// classified against t' = t restricted to X_t as supported (A is a cluster of t'), conflicting (A overlaps a cluster
// of t' without nesting), permitted (neither) or irrelevant (|A| < 2 or A = X_t).
//
// One CTA per source tree.  Both trees become orders of the same k = |X_t| leaves:
//   S-rank r   position of a leaf of X_t in S's depth-first leaf order: a bitmap over S's leaf positions in shared
//              memory plus a prefix of its word popcounts gives the rank of any S leaf position in O(1), so the
//              clade of S-node u is the S-rank range [rank(first leaf of u), rank(one past its last leaf));
//   q          position in t's leaf tour with the other taxa dropped (the tour of t'); td[q] = depth in t of the
//              LCA of t'-neighbours q and q + 1 (range-min of t's tour depths between them), kept in a sparse table.
// For A = S-ranks [a, b):  lo / hi = min / max of q over A and d = min td[lo, hi) = depth of v = LCA_t(A).  A is a
// union of whole children of v (compatible with t') iff every t'-edge with exactly one end in A lies at depth <= d,
// and it is v's own cluster iff moreover it is contiguous in t' with both outer edges above v.  Depths are compared,
// never counted, so unary nodes and polytomies of t need no special case.  The per-clade loop is O(|A|): the work of
// a tree is bounded by the sum over its shared taxa of their depth in S.
//
// The class of every (tree, node) pair goes to a byte matrix; a second kernel sums it per node over the trees in
// tree order, so the weighted sums are the same bits on every run.  Trees are processed in chunks that bound the
// matrix and the per-tree scratch.

#include <algorithm>
#include <climits>
#include <cmath>
#include <vector>

#include "devforest.cuh"
#include "forest.hpp"
#include "supertree.cuh"

namespace scs {
namespace {

constexpr int kThreads = 256;
constexpr uint8_t kSupport = 0, kConflict = 1, kPermitted = 2, kIrrelevant = 3;
constexpr size_t kClassBytes = size_t(256) << 20;     // class matrix of one chunk
constexpr size_t kScratchBytes = size_t(1024) << 20;  // per-tree scratch of one chunk

struct SupportArgs {
    // supertree in depth-first pre-order
    int32_t n_nodes, n_leaves, words, taxa;
    const int32_t *s_parent, *s_first, *s_count;  // parent, first leaf position, leaves below
    const int32_t *pos;                           // taxon -> leaf position in S, -1 if S lacks it
    // source forest and its tours (weighting one)
    const int64_t *tree_off, *leaf_off;
    const int32_t *f_parent, *f_size, *f_taxon, *leaf_taxon, *adj_depth;
    // the chunk
    int32_t t0;
    int64_t leaf0, node0, chunk_leaves;
    int32_t *qpos, *sq, *sr, *table, *kn;
    uint8_t *cls;
    int32_t *per_tree;
};

__global__ void __launch_bounds__(kThreads) sp_tree(SupportArgs a) {
    extern __shared__ uint32_t smem[];
    uint32_t *bits = smem;
    int32_t *wpre = reinterpret_cast<int32_t *>(smem + a.words);
    __shared__ int32_t sums[33];
    __shared__ int32_t tally[3];  // source clusters, supertree clusters, shared
    const int tr = blockIdx.x, t = a.t0 + tr;
    const int64_t nb = a.tree_off[t], lb = a.leaf_off[t];
    const int nn = static_cast<int>(a.tree_off[t + 1] - nb), nl = static_cast<int>(a.leaf_off[t + 1] - lb);
    const int64_t rel = lb - a.leaf0;
    int32_t *qp = a.qpos + rel;
    const int32_t *lt = a.leaf_taxon + lb, *ad = a.adj_depth + lb;
    uint8_t *row = a.cls + static_cast<size_t>(tr) * a.n_nodes;
    auto pos_of = [&](int x) { return x >= 0 && x < a.taxa ? a.pos[x] : -1; };

    for (int w = threadIdx.x; w < a.words; w += blockDim.x) bits[w] = 0;
    if (threadIdx.x < 3) tally[threadIdx.x] = 0;
    __syncthreads();
    for (int j = threadIdx.x; j < nl; j += blockDim.x) {
        const int p = pos_of(lt[j]);
        qp[j] = p >= 0;
        if (p >= 0) atomicOr(&bits[p >> 5], 1u << (p & 31));
    }
    __syncthreads();
    const int k = block_scan(qp, nl, sums);  // qp[j] = t' position of tour position j if it is kept
    if (k < 2) {
        for (int u = threadIdx.x; u < a.n_nodes; u += blockDim.x) row[u] = kIrrelevant;
        if (threadIdx.x < 4) a.per_tree[4 * static_cast<int64_t>(t) + threadIdx.x] = 0;
        return;
    }
    auto kept = [&](int j) { return (j + 1 < nl ? qp[j + 1] : k) > qp[j]; };
    for (int w = threadIdx.x; w < a.words; w += blockDim.x) wpre[w] = __popc(bits[w]);
    __syncthreads();
    block_scan(wpre, a.words, sums);
    auto rank = [&](int p) { return p >= a.n_leaves ? k : bitmap_rank(bits, wpre, p); };

    int32_t *sq = a.sq + rel, *sr = a.sr + rel, *td = a.table + rel;
    for (int j = threadIdx.x; j < nl; j += blockDim.x) {
        if (!kept(j)) continue;
        const int q = qp[j], r = rank(pos_of(lt[j]));
        sq[r] = q;
        sr[q] = r;
        if (q < k - 1) {
            int m = ad[j];
            for (int j2 = j + 1; !kept(j2); ++j2) m = min(m, ad[j2]);
            td[q] = m;
        }
    }
    // sparse table over td[0, k - 1): level l at td + l * chunk_leaves holds the minima of 2^l consecutive entries
    const int edges = k - 1;
    for (int l = 1; (1 << l) <= edges; ++l) {
        __syncthreads();
        const int32_t *below = td + (l - 1) * a.chunk_leaves;
        int32_t *level = td + l * a.chunk_leaves;
        const int half = 1 << (l - 1);
        for (int i = threadIdx.x; i + (1 << l) <= edges; i += blockDim.x) level[i] = min(below[i], below[i + half]);
    }
    __syncthreads();
    auto range_min = [&](int lo, int hi) {  // min td[lo, hi], lo <= hi
        const int l = 31 - __clz(hi - lo + 1);
        const int32_t *level = td + l * a.chunk_leaves;
        return min(level[lo], level[hi - (1 << l) + 1]);
    };

    // |C(t')|: nodes of t whose kept tips are a non-trivial set different from their parent's
    int32_t *kn = a.kn + (nb - a.node0) + tr;  // nn + 1 entries per tree
    for (int v = threadIdx.x; v <= nn; v += blockDim.x) kn[v] = v < nn && pos_of(a.f_taxon[nb + v]) >= 0;
    __syncthreads();
    block_scan(kn, nn + 1, sums);
    {
        int mine = 0;
        for (int v = threadIdx.x; v < nn; v += blockDim.x) {
            const int c = kn[v + a.f_size[nb + v]] - kn[v];
            if (c < 2 || c >= k) continue;
            const int p = a.f_parent[nb + v];
            if (c < kn[p + a.f_size[nb + p]] - kn[p]) ++mine;
        }
        if (mine) atomicAdd(&tally[0], mine);
    }

    int clusters = 0, shared = 0;
    for (int u = threadIdx.x; u < a.n_nodes; u += blockDim.x) {
        const int first = a.s_first[u], count = a.s_count[u];
        const int lo_r = rank(first), hi_r = rank(first + count), m = hi_r - lo_r;
        if (count < 2 || m < 2 || m == k) {
            row[u] = kIrrelevant;
            continue;
        }
        int lo = INT_MAX, hi = -1;
        for (int r = lo_r; r < hi_r; ++r) {
            const int q = sq[r];
            lo = min(lo, q);
            hi = max(hi, q);
        }
        const int d = range_min(lo, hi - 1);
        const int left = lo > 0 ? td[lo - 1] : -1, right = hi < k - 1 ? td[hi] : -1;
        uint8_t c;
        if (left > d || right > d) {
            c = kConflict;
        } else if (hi - lo + 1 == m) {
            c = left < d && right < d ? kSupport : kPermitted;
        } else {
            c = kPermitted;
            for (int r = lo_r; r < hi_r && c == kPermitted; ++r) {
                const int q = sq[r];
                if (q > lo && (sr[q - 1] < lo_r || sr[q - 1] >= hi_r) && td[q - 1] > d) c = kConflict;
                if (q < hi && (sr[q + 1] < lo_r || sr[q + 1] >= hi_r) && td[q] > d) c = kConflict;
            }
        }
        row[u] = c;
        const int pu = a.s_parent[u];  // u is not the root: the root's clade is X_t
        if (m < rank(a.s_first[pu] + a.s_count[pu]) - rank(a.s_first[pu])) {
            ++clusters;
            shared += c == kSupport;
        }
    }
    if (clusters) atomicAdd(&tally[1], clusters);
    if (shared) atomicAdd(&tally[2], shared);
    __syncthreads();
    if (threadIdx.x == 0) {
        int32_t *out = a.per_tree + 4 * static_cast<int64_t>(t);
        out[0] = tally[2];
        out[1] = tally[0];
        out[2] = tally[1];
        out[3] = tally[0] + tally[1] - 2 * tally[2];
    }
}

// counts[3u + c] += 1 and weighted[3u + c] += weight of the tree, over the chunk's trees in order (one thread per node)
__global__ void sp_reduce(int n_nodes, int trees, const uint8_t *__restrict__ cls, const double *__restrict__ weight,
                          int32_t *__restrict__ counts, double *__restrict__ weighted) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= n_nodes) return;
    int32_t cnt[3] = {counts[3 * u], counts[3 * u + 1], counts[3 * u + 2]};
    double sum[3] = {weighted[3 * u], weighted[3 * u + 1], weighted[3 * u + 2]};
    for (int t = 0; t < trees; ++t) {
        const int c = cls[static_cast<size_t>(t) * n_nodes + u];
        if (c == kIrrelevant) continue;
        cnt[c] += 1;
        sum[c] += weight[t];
    }
    for (int c = 0; c < 3; ++c) {
        counts[3 * u + c] = cnt[c];
        weighted[3 * u + c] = sum[c];
    }
}

}  // namespace
}  // namespace scs

using namespace scs;

extern "C" int scs_supertree_support(scs_ctx *ctx, const scs_forest *sources, int64_t num_nodes, const int32_t *parent,
                                     const int32_t *taxon, int32_t *counts, double *weighted, int32_t *per_tree) {
    if (!ctx) return SCS_ERR_INVALID;
    if (!sources || !parent || !taxon || !counts || !per_tree || num_nodes <= 0 || num_nodes >= (int64_t(1) << 31))
        return fail(ctx, SCS_ERR_INVALID, "scs_supertree_support: bad argument");
    const int taxa = sources->num_taxa;
    PreorderTree s;
    if (preorder_supertree(num_nodes, parent, taxon, taxa, &s))
        return fail(ctx, SCS_ERR_INPUT, "scs_supertree_support: malformed supertree (parent[i] >= i, a tip without a "
                                        "taxon of the forest, or a repeated taxon)");
    const int n = static_cast<int>(num_nodes), T = sources->num_trees();
    const int words = (s.leaves + 31) / 32;
    const size_t smem = static_cast<size_t>(words) * 8;
    if (smem + 1024 > ctx->smem_optin)  // room for the static shared arrays
        return fail(ctx, SCS_ERR_INVALID, "scs_supertree_support: the supertree has too many tips for the shared-memory bitmap");
    std::fill(counts, counts + 3 * num_nodes, 0);
    if (weighted) std::fill(weighted, weighted + 3 * num_nodes, 0.0);
    if (T == 0) return SCS_OK;

    // chunks of trees: the class matrix and the per-tree scratch stay bounded
    const std::vector<int64_t> &loff = sources->leaf_offsets, &noff = sources->node_offsets;
    int64_t max_leaves = 0;
    for (int t = 0; t < T; ++t) max_leaves = std::max(max_leaves, loff[t + 1] - loff[t]);
    int levels = 1;
    while ((int64_t(1) << levels) <= max_leaves) ++levels;
    std::vector<int> chunk_begin{0};
    int64_t most_leaves = 0, most_nodes = 0, most_trees = 0;
    for (int t = 0; t < T;) {
        const int b = chunk_begin.back();
        int e = t + 1;
        while (e < T && static_cast<size_t>(e + 1 - b) * n <= kClassBytes &&
               static_cast<size_t>(loff[e + 1] - loff[b]) * (levels + 3) * 4 <= kScratchBytes)
            ++e;
        most_leaves = std::max(most_leaves, loff[e] - loff[b]);
        most_nodes = std::max(most_nodes, noff[e] - noff[b]);
        most_trees = std::max<int64_t>(most_trees, e - b);
        chunk_begin.push_back(e);
        t = e;
    }

    DevForest forest;
    DevTours tours;
    GrowBuf ident, flags, s_parent, s_first, s_count, pos, qpos, sq, sr, table, kn, cls, weight, d_counts, d_weighted, d_per_tree;
    auto cleanup = [&] {
        forest.free_all(ctx);
        tours.free_all(ctx);
        for (GrowBuf *b : {&ident, &flags, &s_parent, &s_first, &s_count, &pos, &qpos, &sq, &sr, &table, &kn, &cls, &weight,
                           &d_counts, &d_weighted, &d_per_tree})
            release(ctx, *b);
        cudaStreamSynchronize(ctx->stream);
    };
    auto run = [&]() -> int {
        int rc;
        if ((rc = devforest_upload(ctx, sources, 0, &forest))) return rc;
        std::vector<int32_t> identity(static_cast<size_t>(taxa > 0 ? taxa : 1));
        for (size_t x = 0; x < identity.size(); ++x) identity[x] = static_cast<int32_t>(x);
        auto put = [&](GrowBuf &buf, const void *src, size_t bytes) -> int {
            int r;
            if ((r = grow(ctx, buf, bytes))) return r;
            SCS_CUDA(ctx, cudaMemcpyAsync(buf.ptr, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
            return SCS_OK;
        };
        const size_t nb = static_cast<size_t>(n) * sizeof(int32_t);
        if ((rc = put(ident, identity.data(), identity.size() * sizeof(int32_t)))) return rc;
        if ((rc = put(s_parent, s.parent.data(), nb)) || (rc = put(s_first, s.first.data(), nb)) ||
            (rc = put(s_count, s.count.data(), nb)) || (rc = put(pos, s.pos.data(), s.pos.size() * sizeof(int32_t))) ||
            (rc = put(weight, sources->weight.data(), static_cast<size_t>(T) * sizeof(double))))
            return rc;
        if ((rc = grow(ctx, flags, 2 * sizeof(int32_t)))) return rc;
        SCS_CUDA(ctx, cudaMemsetAsync(flags.ptr, 0, 2 * sizeof(int32_t), ctx->stream));
        if ((rc = devforest_tours(ctx, forest, 0, ident.as<int32_t>(), &tours, flags.as<int32_t>()))) return rc;
        const size_t L = static_cast<size_t>(most_leaves) + 1;
        if ((rc = grow(ctx, qpos, L * 4)) || (rc = grow(ctx, sq, L * 4)) || (rc = grow(ctx, sr, L * 4)) ||
            (rc = grow(ctx, table, L * levels * 4)) || (rc = grow(ctx, kn, static_cast<size_t>(most_nodes + most_trees) * 4)) ||
            (rc = grow(ctx, cls, static_cast<size_t>(most_trees) * n)) || (rc = grow(ctx, d_counts, 3 * nb)) ||
            (rc = grow(ctx, d_weighted, 3 * static_cast<size_t>(n) * sizeof(double))) ||
            (rc = grow(ctx, d_per_tree, 4 * static_cast<size_t>(T) * sizeof(int32_t))))
            return rc;
        SCS_CUDA(ctx, cudaMemsetAsync(d_counts.ptr, 0, 3 * nb, ctx->stream));
        SCS_CUDA(ctx, cudaMemsetAsync(d_weighted.ptr, 0, 3 * static_cast<size_t>(n) * sizeof(double), ctx->stream));
        if (smem > 48 * 1024) SCS_CUDA(ctx, cudaFuncSetAttribute(sp_tree, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));

        SupportArgs args{};
        args.n_nodes = n;
        args.n_leaves = s.leaves;
        args.words = words;
        args.taxa = taxa;
        args.s_parent = s_parent.as<int32_t>();
        args.s_first = s_first.as<int32_t>();
        args.s_count = s_count.as<int32_t>();
        args.pos = pos.as<int32_t>();
        args.tree_off = forest.tree_off.as<int64_t>();
        args.leaf_off = forest.leaf_off.as<int64_t>();
        args.f_parent = forest.parent.as<int32_t>();
        args.f_size = forest.size.as<int32_t>();
        args.f_taxon = forest.taxon.as<int32_t>();
        args.leaf_taxon = tours.leaf_taxon.as<int32_t>();
        args.adj_depth = tours.adj_depth.as<int32_t>();
        args.chunk_leaves = static_cast<int64_t>(L);
        args.qpos = qpos.as<int32_t>();
        args.sq = sq.as<int32_t>();
        args.sr = sr.as<int32_t>();
        args.table = table.as<int32_t>();
        args.kn = kn.as<int32_t>();
        args.cls = cls.as<uint8_t>();
        args.per_tree = d_per_tree.as<int32_t>();
        for (size_t c = 0; c + 1 < chunk_begin.size(); ++c) {
            const int b = chunk_begin[c], e = chunk_begin[c + 1];
            args.t0 = b;
            args.leaf0 = loff[b];
            args.node0 = noff[b];
            sp_tree<<<e - b, kThreads, smem, ctx->stream>>>(args);
            SCS_LAUNCHED(ctx, "sp_tree");
            sp_reduce<<<ceil_div(n, 256), 256, 0, ctx->stream>>>(n, e - b, cls.as<uint8_t>(), weight.as<double>() + b,
                                                                 d_counts.as<int32_t>(), d_weighted.as<double>());
            SCS_LAUNCHED(ctx, "sp_reduce");
        }
        std::vector<int32_t> cnt(3 * static_cast<size_t>(n));
        std::vector<double> wsum(3 * static_cast<size_t>(n));
        SCS_CUDA(ctx, cudaMemcpyAsync(cnt.data(), d_counts.ptr, 3 * nb, cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaMemcpyAsync(wsum.data(), d_weighted.ptr, wsum.size() * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaMemcpyAsync(per_tree, d_per_tree.ptr, 4 * static_cast<size_t>(T) * sizeof(int32_t),
                                      cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        ctx->d2h_bytes += static_cast<int64_t>(3 * nb + wsum.size() * sizeof(double) + 4 * static_cast<size_t>(T) * 4);
        for (int u = 0; u < n; ++u) {
            const int32_t v = s.order[u];
            for (int c = 0; c < 3; ++c) {
                counts[3 * static_cast<int64_t>(v) + c] = cnt[3 * static_cast<size_t>(u) + c];
                if (weighted) weighted[3 * static_cast<int64_t>(v) + c] = wsum[3 * static_cast<size_t>(u) + c];
            }
        }
        return SCS_OK;
    };
    const int rc = run();
    cleanup();
    return rc;
}
