// Rooted triplet fit of a supertree (scs_supertree_triplets): for every source tree t with k = |X_t| shared taxa,
// how many three-taxon statements of X_t the restricted source tree t' = t|X_t resolves, how many the restricted
// supertree s' = S|X_t resolves, and how many of them the two resolve the same way (agree) or differently (contradict).
//
// Counting identity.  Fix a taxon a of X_t; for x in X_t \ {a} let alpha(x) = depth in t of LCA_t(a, x) and
// beta(x) = depth in S of LCA_S(a, x).  Restriction keeps the order of the ancestors of a, so depths of the
// unrestricted trees compare correctly.  {a, b, x} is ab|x in t iff alpha(x) < alpha(b), and in S iff beta(x) <
// beta(b).  Summed over all rows a, the unordered pairs {b, x} with
//   alpha different                               count every resolved source triplet twice,
//   beta different                                count every resolved supertree triplet twice,
//   alpha and beta both ordered the same way      count every agreeing triplet twice,
//   alpha and beta both ordered the opposite way  count every contradicting triplet once
// (ab|x against ax|b is seen from row a only: from row b the supertree depths tie).
//
// One warp per row a.  The tree's shared taxa in the order of t's leaf tour form the tour of t'; td[q] = depth in t
// of the LCA of t'-neighbours q and q + 1.  alpha is a running minimum of td outward from a, so {x : alpha(x) >= d}
// is a window of the tour of t' around a.  The warp grows that window one depth level at a time, deepest first; the
// taxa a level adds are counted against those already inside (all of them deeper in t) with a Fenwick tree over
// beta in shared memory, then added to it.  beta(x) is an O(1) range minimum over S's leaf order (a sparse table of
// the depths between consecutive leaves of S, built once).  A row costs O(k log D + D / 32) for a supertree of
// depth D, a tree O(k^2 log D + k D / 32).
//
// Integer counts are exact; every row writes its own partial counts and a second kernel adds a tree's rows in tour
// order.  Trees are processed in chunks that bound the per-leaf scratch.

#include <algorithm>
#include <vector>

#include "devforest.cuh"
#include "forest.hpp"
#include "supertree.cuh"

namespace scs {
namespace {

constexpr int kPrepThreads = 256;
constexpr int kMaxRowWarps = 8;
constexpr size_t kScratchBytes = size_t(1024) << 20;         // per-leaf scratch of one chunk
constexpr size_t kLeafScratch = 3 * sizeof(int32_t) + 4 * sizeof(int64_t);  // qpos, spos, td + four row counts

struct TripletArgs {
    // supertree: taxon -> leaf position (-1 if S lacks it), depth of every leaf, sparse table over the depths of the
    // LCAs of consecutive leaves (level l at stab + l * n_leaves)
    int32_t taxa, n_leaves;
    const int32_t *pos, *leaf_depth, *stab;
    // source forest and its tours (weighting one)
    const int64_t *leaf_off;
    const int32_t *leaf_taxon, *adj_depth;
    // the chunk: trees [t0, t1), tour positions [leaf0, leaf0 + chunk_leaves)
    int32_t t0, t1;
    int64_t leaf0, chunk_leaves;
    int32_t *qpos;   // [chunk leaves]: exclusive scan of "shared with S" over the tour = t' position
    int32_t *spos;   // [chunk leaves]: per tree, at its first tour position: S leaf position of t' position q
    int32_t *td;     // [chunk leaves]: per tree, likewise: depth in t of the LCA of t' positions q and q + 1
    int32_t *k;      // [chunk trees]
    int64_t *rows;   // [chunk leaves][4]: per row a: R1, R2, AG, CO
    int64_t *per_tree;
};

// One CTA per tree: t' positions, the S positions of its taxa and the depths between t'-neighbours.
__global__ void __launch_bounds__(kPrepThreads) tp_prep(TripletArgs a) {
    __shared__ int32_t sums[33];
    const int t = a.t0 + blockIdx.x;
    const int64_t lb = a.leaf_off[t];
    const int nl = static_cast<int>(a.leaf_off[t + 1] - lb);
    const int64_t rel = lb - a.leaf0;
    int32_t *qp = a.qpos + rel;
    const int32_t *lt = a.leaf_taxon + lb, *ad = a.adj_depth + lb;
    auto pos_of = [&](int x) { return x >= 0 && x < a.taxa ? a.pos[x] : -1; };
    for (int j = threadIdx.x; j < nl; j += blockDim.x) qp[j] = pos_of(lt[j]) >= 0;
    __syncthreads();
    const int k = block_scan(qp, nl, sums);
    if (threadIdx.x == 0) a.k[blockIdx.x] = k;
    int32_t *sp = a.spos + rel, *td = a.td + rel;
    for (int j = threadIdx.x; j < nl; j += blockDim.x) {
        const int q = qp[j];
        if ((j + 1 < nl ? qp[j + 1] : k) == q) continue;  // not shared
        sp[q] = pos_of(lt[j]);
        if (q < k - 1) {
            int m = ad[j];
            for (int j2 = j + 1; (j2 + 1 < nl ? qp[j2 + 1] : k) == qp[j2]; ++j2) m = min(m, ad[j2]);
            td[q] = m;
        }
    }
}

// depth in S of the LCA of the leaves at S positions p != r
__device__ __forceinline__ int s_lca_depth(const TripletArgs &a, int p, int r) {
    const int lo = min(p, r), hi = max(p, r);
    const int l = 31 - __clz(hi - lo);
    const int32_t *level = a.stab + static_cast<int64_t>(l) * a.n_leaves;
    return min(__ldg(level + lo), __ldg(level + hi - (1 << l)));
}

// One warp per row: tour position g of the chunk.  Shared memory per warp: Fenwick tree over beta + 1 in [1, m] and
// a histogram of beta in [0, m), m = depth of a in S (beta < m).
__global__ void __launch_bounds__(kMaxRowWarps * 32, 1) tp_rows(TripletArgs a, int stride) {
    extern __shared__ int32_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t g = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + warp;
    if (g >= a.chunk_leaves) return;
    int64_t *out = a.rows + 4 * g;
    int lo = a.t0, hi = a.t1;  // the tree of g: the last t with leaf_off[t] <= leaf0 + g
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (a.leaf_off[mid] <= a.leaf0 + g) lo = mid; else hi = mid;
    }
    const int64_t rel = a.leaf_off[lo] - a.leaf0;
    const int nl = static_cast<int>(a.leaf_off[lo + 1] - a.leaf_off[lo]), j = static_cast<int>(g - rel);
    const int k = a.k[lo - a.t0];
    const int32_t *qp = a.qpos + rel;
    const int qa = qp[j];
    if (k < 3 || (j + 1 < nl ? qp[j + 1] : k) == qa) {  // fewer than three shared taxa, or a is not shared
        if (lane < 4) out[lane] = 0;
        return;
    }
    const int32_t *sp = a.spos + rel, *td = a.td + rel;
    const int pa = sp[qa], m = a.leaf_depth[pa];
    int32_t *fw = smem + warp * 2 * stride, *hist = fw + stride;
    for (int i = lane; i <= m; i += 32) fw[i] = 0;
    for (int i = lane; i < m; i += 32) hist[i] = 0;
    __syncwarp();

    long long r1 = 0, ag = 0, co = 0;
    int L = qa, R = qa, inside = 0;  // t' positions [L, R] are inside the window (a itself is no point)
    for (;;) {
        const int eL = L > 0 ? td[L - 1] : -1, eR = R < k - 1 ? td[R] : -1;
        const int level = max(eL, eR);
        if (level < 0) break;
        int nL = L, nR = R;
        if (eL == level) {  // q joins while td[q .. L - 1] >= level
            for (;;) {
                const int q = nL - 1 - lane;
                const unsigned bad = __ballot_sync(0xffffffffu, !(q >= 0 && td[q] >= level));
                const int run = bad ? __ffs(bad) - 1 : 32;
                nL -= run;
                if (run < 32) break;
            }
        }
        if (eR == level) {  // q joins while td[R .. q - 1] >= level
            for (;;) {
                const int q = nR + 1 + lane;
                const unsigned bad = __ballot_sync(0xffffffffu, !(q < k && td[q - 1] >= level));
                const int run = bad ? __ffs(bad) - 1 : 32;
                nR += run;
                if (run < 32) break;
            }
        }
        const int left = L - nL, added = left + nR - R;
        // the new taxa x (alpha(x) = level) against the y inside (alpha(y) > level): concordant when beta(y) >
        // beta(x), discordant when beta(y) < beta(x)
        for (int i = lane; i < added; i += 32) {
            const int b = s_lca_depth(a, pa, sp[i < left ? nL + i : R + 1 + (i - left)]);
            int below = 0;
            for (int f = b; f > 0; f -= f & -f) below += fw[f];
            co += below;
            ag += inside - below - hist[b];
        }
        __syncwarp();
        for (int i = lane; i < added; i += 32) {
            const int b = s_lca_depth(a, pa, sp[i < left ? nL + i : R + 1 + (i - left)]);
            for (int f = b + 1; f <= m; f += f & -f) atomicAdd(&fw[f], 1);
            atomicAdd(&hist[b], 1);
        }
        __syncwarp();
        if (lane == 0) r1 += static_cast<long long>(inside) * added;
        inside += added;
        L = nL;
        R = nR;
    }
    long long ties = 0;  // pairs {b, x} with beta(b) = beta(x)
    for (int i = lane; i < m; i += 32) ties += static_cast<long long>(hist[i]) * (hist[i] - 1) / 2;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        r1 += __shfl_down_sync(0xffffffffu, r1, off);
        ag += __shfl_down_sync(0xffffffffu, ag, off);
        co += __shfl_down_sync(0xffffffffu, co, off);
        ties += __shfl_down_sync(0xffffffffu, ties, off);
    }
    if (lane == 0) {
        out[0] = r1;
        out[1] = static_cast<long long>(k - 1) * (k - 2) / 2 - ties;
        out[2] = ag;
        out[3] = co;
    }
}

// One warp per tree of the chunk: its rows summed in tour order.
__global__ void tp_reduce(TripletArgs a) {
    const int64_t w = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= a.t1 - a.t0) return;
    const int t = a.t0 + static_cast<int>(w);
    const int64_t b = a.leaf_off[t] - a.leaf0, e = a.leaf_off[t + 1] - a.leaf0;
    long long s[4] = {0, 0, 0, 0};
    for (int64_t g = b + lane; g < e; g += 32)
        for (int c = 0; c < 4; ++c) s[c] += a.rows[4 * g + c];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1)
        for (int c = 0; c < 4; ++c) s[c] += __shfl_down_sync(0xffffffffu, s[c], off);
    if (lane == 0) {
        int64_t *o = a.per_tree + 5 * static_cast<int64_t>(t);
        o[0] = a.k[w];
        o[1] = s[0] / 2;  // resolved in t'
        o[2] = s[1] / 2;  // resolved in s'
        o[3] = s[2] / 2;  // agree
        o[4] = s[3];      // contradict
    }
}

}  // namespace
}  // namespace scs

using namespace scs;

extern "C" int scs_supertree_triplets(scs_ctx *ctx, const scs_forest *sources, int64_t num_nodes, const int32_t *parent,
                                      const int32_t *taxon, int64_t *per_tree) {
    if (!ctx) return SCS_ERR_INVALID;
    if (!sources || !parent || !taxon || !per_tree || num_nodes <= 0 || num_nodes >= (int64_t(1) << 31))
        return fail(ctx, SCS_ERR_INVALID, "scs_supertree_triplets: bad argument");
    const int taxa = sources->num_taxa;
    PreorderTree s;
    if (preorder_supertree(num_nodes, parent, taxon, taxa, &s))
        return fail(ctx, SCS_ERR_INPUT, "scs_supertree_triplets: malformed supertree (parent[i] >= i, a tip without a "
                                        "taxon of the forest, or a repeated taxon)");
    const int n = static_cast<int>(num_nodes), T = sources->num_trees(), NL = s.leaves;
    // depth of every leaf and of the LCA of consecutive leaves: in pre-order the node after a tip hangs off that LCA
    std::vector<int32_t> depth(static_cast<size_t>(n), 0), leaf_depth(static_cast<size_t>(NL), 0);
    std::vector<int32_t> adj(static_cast<size_t>(std::max(NL - 1, 1)), 0);
    int max_depth = 0;
    for (int u = 1; u < n; ++u) depth[u] = depth[s.parent[u]] + 1;
    for (int u = 0; u < n; ++u) {
        if (u + 1 < n && s.parent[u + 1] == u) continue;  // not a tip
        leaf_depth[s.first[u]] = depth[u];
        max_depth = std::max(max_depth, depth[u]);
        if (u + 1 < n) adj[s.first[u]] = depth[s.parent[u + 1]];
    }
    int levels = 1;
    while ((int64_t(1) << levels) <= NL - 1) ++levels;
    std::vector<int32_t> stab(static_cast<size_t>(levels) * NL, 0);
    std::copy(adj.begin(), adj.begin() + std::max(NL - 1, 0), stab.begin());
    for (int l = 1; l < levels; ++l)
        for (int i = 0; i + (1 << l) <= NL - 1; ++i)
            stab[static_cast<size_t>(l) * NL + i] = std::min(stab[static_cast<size_t>(l - 1) * NL + i],
                                                             stab[static_cast<size_t>(l - 1) * NL + i + (1 << (l - 1))]);
    // per row warp: a Fenwick tree (max_depth + 1 ints) and a histogram (max_depth ints) in shared memory
    const int stride = max_depth + 1;
    const size_t warp_smem = 2 * static_cast<size_t>(stride) * sizeof(int32_t);
    const int warps = static_cast<int>(std::min<size_t>(kMaxRowWarps, ctx->smem_optin / warp_smem));
    if (warps < 1)
        return fail(ctx, SCS_ERR_INVALID, "scs_supertree_triplets: the supertree is too deep for the shared-memory "
                                          "Fenwick tree of a row");
    std::fill(per_tree, per_tree + 5 * static_cast<int64_t>(T), 0);
    if (T == 0) return SCS_OK;

    const std::vector<int64_t> &loff = sources->leaf_offsets;
    std::vector<int> chunk_begin{0};
    int64_t most_leaves = 0, most_trees = 0;
    for (int t = 0; t < T;) {
        const int b = chunk_begin.back();
        int e = t + 1;
        while (e < T && static_cast<size_t>(loff[e + 1] - loff[b]) * kLeafScratch <= kScratchBytes) ++e;
        most_leaves = std::max(most_leaves, loff[e] - loff[b]);
        most_trees = std::max<int64_t>(most_trees, e - b);
        chunk_begin.push_back(e);
        t = e;
    }

    DevForest forest;
    DevTours tours;
    GrowBuf ident, flags, pos, d_leaf_depth, d_stab, qpos, spos, td, kbuf, rows, d_per_tree;
    auto cleanup = [&] {
        forest.free_all(ctx);
        tours.free_all(ctx);
        for (GrowBuf *b : {&ident, &flags, &pos, &d_leaf_depth, &d_stab, &qpos, &spos, &td, &kbuf, &rows, &d_per_tree})
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
        if ((rc = put(ident, identity.data(), identity.size() * sizeof(int32_t))) ||
            (rc = put(pos, s.pos.data(), s.pos.size() * sizeof(int32_t))) ||
            (rc = put(d_leaf_depth, leaf_depth.data(), leaf_depth.size() * sizeof(int32_t))) ||
            (rc = put(d_stab, stab.data(), stab.size() * sizeof(int32_t))))
            return rc;
        if ((rc = grow(ctx, flags, 2 * sizeof(int32_t)))) return rc;
        SCS_CUDA(ctx, cudaMemsetAsync(flags.ptr, 0, 2 * sizeof(int32_t), ctx->stream));
        if ((rc = devforest_tours(ctx, forest, 0, ident.as<int32_t>(), &tours, flags.as<int32_t>()))) return rc;
        const size_t L = static_cast<size_t>(most_leaves) + 1;
        if ((rc = grow(ctx, qpos, L * 4)) || (rc = grow(ctx, spos, L * 4)) || (rc = grow(ctx, td, L * 4)) ||
            (rc = grow(ctx, rows, L * 4 * sizeof(int64_t))) || (rc = grow(ctx, kbuf, static_cast<size_t>(most_trees) * 4)) ||
            (rc = grow(ctx, d_per_tree, 5 * static_cast<size_t>(T) * sizeof(int64_t))))
            return rc;
        const size_t row_smem = static_cast<size_t>(warps) * warp_smem;
        if (row_smem > 48 * 1024)
            SCS_CUDA(ctx, cudaFuncSetAttribute(tp_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(row_smem)));

        TripletArgs args{};
        args.taxa = taxa;
        args.n_leaves = NL;
        args.pos = pos.as<int32_t>();
        args.leaf_depth = d_leaf_depth.as<int32_t>();
        args.stab = d_stab.as<int32_t>();
        args.leaf_off = forest.leaf_off.as<int64_t>();
        args.leaf_taxon = tours.leaf_taxon.as<int32_t>();
        args.adj_depth = tours.adj_depth.as<int32_t>();
        args.qpos = qpos.as<int32_t>();
        args.spos = spos.as<int32_t>();
        args.td = td.as<int32_t>();
        args.k = kbuf.as<int32_t>();
        args.rows = rows.as<int64_t>();
        args.per_tree = d_per_tree.as<int64_t>();
        for (size_t c = 0; c + 1 < chunk_begin.size(); ++c) {
            const int b = chunk_begin[c], e = chunk_begin[c + 1];
            args.t0 = b;
            args.t1 = e;
            args.leaf0 = loff[b];
            args.chunk_leaves = loff[e] - loff[b];
            tp_prep<<<e - b, kPrepThreads, 0, ctx->stream>>>(args);
            SCS_LAUNCHED(ctx, "tp_prep");
            if (args.chunk_leaves > 0) {
                tp_rows<<<ceil_div(args.chunk_leaves, warps), warps * 32, row_smem, ctx->stream>>>(args, stride);
                SCS_LAUNCHED(ctx, "tp_rows");
            }
            tp_reduce<<<ceil_div(e - b, 8), 256, 0, ctx->stream>>>(args);
            SCS_LAUNCHED(ctx, "tp_reduce");
        }
        const size_t out_bytes = 5 * static_cast<size_t>(T) * sizeof(int64_t);
        SCS_CUDA(ctx, cudaMemcpyAsync(per_tree, d_per_tree.ptr, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        ctx->d2h_bytes += static_cast<int64_t>(out_bytes);
        // a lone tip has no tour: it shares one taxon with S or none
        const std::vector<int64_t> &noff = sources->node_offsets;
        for (int t = 0; t < T; ++t)
            if (noff[t + 1] - noff[t] == 1) {
                const int x = sources->taxon[noff[t]];
                per_tree[5 * static_cast<int64_t>(t)] = x >= 0 && x < taxa && s.pos[x] >= 0;
            }
        return SCS_OK;
    };
    const int rc = run();
    cleanup();
    return rc;
}
