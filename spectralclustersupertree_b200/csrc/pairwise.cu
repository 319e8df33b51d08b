// Rooted Robinson-Foulds distances between every pair of source trees on the taxa they share
// (scs_forest_pairwise_rf).  For trees t_i, t_j with X = X_ij = taxa(t_i) & taxa(t_j), k = |X|: the number of
// non-trivial clusters (2 <= |c| < k) of t_i|X and of t_j|X, and how many of them the two have in common.
//
// Pass 1 (pw_bitmap, pw_shared): one bitmap row per tree over the taxa; k_ij is the AND-popcount of rows i and j,
// computed for every pair in 64 x 64 tiles of the upper triangle with both rows' words staged in shared memory.  The
// pairs with k_ij >= 3 (the diagonal included) go to a work list; the others have no non-trivial cluster.
//
// Pass 2 (pw_pairs): one CTA per listed pair, persistent CTAs taking pairs from a counter.  X is the AND of the two
// rows, held in shared memory with the prefix of its word popcounts, so every taxon of X has an O(1) rank r in X.
// Each tree's leaf tour, with the tips outside X dropped, is the tour of its restriction t' (block scan of the kept
// flags: t' position).  The gap g[p] between t'-neighbours p and p + 1 is the depth in t of their LCA: the minimum of
// the tour's adj_depth between the two tips, one range-minimum over a sparse table of the tree's tour (pw_tour_table,
// built once).  Restriction keeps the order of the ancestors of every tip, so depths of the unrestricted tree compare
// correctly, and unary nodes and polytomies need no special case.  t_j's positions go to a rank-indexed array, which
// maps every t_i' position p to the t_j' position qi[p] of the same taxon.
//
// The clusters of t' are the maximal windows of t' positions around a gap p in which every gap is >= g[p].  Gap p
// names its window iff the nearest gap left of it with depth <= g[p] is strictly shallower (or absent); every window
// is named exactly once and windows of different depths are different sets, so the named gaps minus the root window
// count the non-trivial clusters.  Both window ends are binary descents over a sparse table of g (O(log k)).  A window
// [l, r] of t_i' of size m is a cluster of t_j' iff qi[l, r] spans exactly m positions [lo, hi] and, with d = min
// g_j[lo, hi), the outer gaps g_j[lo - 1], g_j[hi] are < d (or absent): range minima and maxima over sparse tables of
// qi and g_j.  A pair costs O(k_i + k_j + k log k) whatever the depth of the trees; every count is an exact integer,
// written to the pair's own entries, so the order in which CTAs take pairs changes no bit.

#include <algorithm>
#include <climits>
#include <vector>

#include "devforest.cuh"
#include "forest.hpp"
#include "supertree.cuh"

namespace scs {
namespace {

constexpr int kThreads = 256;
constexpr int kTile = 64;       // trees per side of a pass-1 tile (16 x 16 threads, 4 x 4 pairs each)
constexpr int kTileWords = 32;  // bitmap words per pass-1 stage
constexpr size_t kScratchBytes = size_t(4096) << 20;  // per-CTA scratch of pass 2, all resident CTAs together

// Row t of the bitmap: bit x set iff tree t has a tip labelled x (rows zeroed beforehand; one CTA per tree).
__global__ void pw_bitmap(const int64_t *__restrict__ tree_off, const int32_t *__restrict__ taxon, int taxa, int words,
                          uint32_t *__restrict__ bits) {
    const int t = blockIdx.x;
    uint32_t *row = bits + static_cast<int64_t>(t) * words;
    for (int64_t v = tree_off[t] + threadIdx.x; v < tree_off[t + 1]; v += blockDim.x) {
        const int x = taxon[v];
        if (x >= 0 && x < taxa) atomicOr(&row[x >> 5], 1u << (x & 31));
    }
}

// shared[i][j] = |taxa(t_i) & taxa(t_j)| for every pair of one tile of the upper triangle (both triangles written);
// the pairs i <= j with k >= 3 are appended to `list`, the largest such k to *max_k.
__global__ void __launch_bounds__(kThreads) pw_shared(int T, int words, const uint32_t *__restrict__ bits,
                                                      int32_t *__restrict__ shared, int2 *__restrict__ list,
                                                      unsigned long long *count, int *max_k) {
    __shared__ uint32_t as[kTile][kTileWords + 1], bs[kTile][kTileWords + 1];
    const int nb = (T + kTile - 1) / kTile;
    int bi = 0, rest = static_cast<int>(blockIdx.x);
    while (rest >= nb - bi) {
        rest -= nb - bi;
        ++bi;
    }
    const int i0 = bi * kTile, j0 = (bi + rest) * kTile;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    int acc[4][4] = {};
    for (int w0 = 0; w0 < words; w0 += kTileWords) {
        for (int e = threadIdx.x; e < kTile * kTileWords; e += kThreads) {
            const int r = e / kTileWords, w = e % kTileWords;
            const bool in = w0 + w < words;
            as[r][w] = in && i0 + r < T ? bits[static_cast<int64_t>(i0 + r) * words + w0 + w] : 0u;
            bs[r][w] = in && j0 + r < T ? bits[static_cast<int64_t>(j0 + r) * words + w0 + w] : 0u;
        }
        __syncthreads();
#pragma unroll 8
        for (int w = 0; w < kTileWords; ++w) {
            uint32_t a[4], b[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) a[r] = as[ty + 16 * r][w];
#pragma unroll
            for (int c = 0; c < 4; ++c) b[c] = bs[tx + 16 * c][w];
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[r][c] += __popc(a[r] & b[c]);
        }
        __syncthreads();
    }
    int mine = 0, kmax = 0;
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int i = i0 + ty + 16 * r, j = j0 + tx + 16 * c;
            if (i >= T || j >= T) continue;
            shared[static_cast<int64_t>(i) * T + j] = acc[r][c];
            shared[static_cast<int64_t>(j) * T + i] = acc[r][c];
            if (i <= j && acc[r][c] >= 3) {
                ++mine;
                kmax = max(kmax, acc[r][c]);
            }
        }
    // one atomic per warp for the list slots
    const int lane = threadIdx.x & 31;
    int incl = mine;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int o = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += o;
    }
    unsigned long long base = 0;
    if (lane == 31 && incl) base = atomicAdd(count, static_cast<unsigned long long>(incl));
    base = __shfl_sync(0xffffffffu, base, 31) + static_cast<unsigned long long>(incl - mine);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, off));
    if (lane == 0 && kmax) atomicMax(max_k, kmax);
    if (!mine) return;
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int i = i0 + ty + 16 * r, j = j0 + tx + 16 * c;
            if (i < T && j < T && i <= j && acc[r][c] >= 3) list[base++] = make_int2(i, j);
        }
}

// Sparse table of the range minima of adj_depth over each tree's tour: level l at table + l * leaves holds the minima
// of 2^l consecutive entries of the same tree (one CTA per tree; level 0 is adj_depth itself).
__global__ void pw_tour_table(const int64_t *__restrict__ leaf_off, int64_t leaves, int32_t *table) {
    const int t = blockIdx.x;
    const int64_t lb = leaf_off[t];
    const int nl = static_cast<int>(leaf_off[t + 1] - lb);
    for (int l = 1; (1 << l) <= nl; ++l) {
        const int32_t *below = table + (l - 1) * leaves + lb;
        int32_t *level = table + l * leaves + lb;
        const int half = 1 << (l - 1);
        for (int i = threadIdx.x; i + (1 << l) <= nl; i += blockDim.x) level[i] = min(below[i], below[i + half]);
        __syncthreads();
    }
}

struct PairArgs {
    int32_t T, words;
    const uint32_t *bits;  // [T][words]
    // the forest's tours (weighting one) and the sparse table over their adj_depth
    const int64_t *leaf_off;
    const int32_t *leaf_taxon, *tour_min;
    int64_t leaves;
    // the work list and the counter the CTAs take pairs from
    const int2 *list;
    int64_t pairs;
    unsigned long long *next;
    // per-CTA scratch: flag [max_leaves + 1], kidx, jpos [max_k], then four tables of `levels` x max_k
    int32_t *scratch;
    int64_t slot, max_leaves, max_k;
    int32_t levels;
    int32_t *clusters, *common;  // [T][T]
};

// min of a sparse table (level l at tab + l * ld) over [lo, hi], lo <= hi; likewise the max
__device__ __forceinline__ int table_min(const int32_t *tab, int64_t ld, int lo, int hi) {
    const int l = 31 - __clz(hi - lo + 1);
    return min(tab[l * ld + lo], tab[l * ld + hi - (1 << l) + 1]);
}
__device__ __forceinline__ int table_max(const int32_t *tab, int64_t ld, int lo, int hi) {
    const int l = 31 - __clz(hi - lo + 1);
    return max(tab[l * ld + lo], tab[l * ld + hi - (1 << l) + 1]);
}

// First tip of the window of gap p (gaps [0, n), min table g) if p names it, else -1: the nearest gap left of p with
// depth <= g[p] must be shallower, or absent.
__device__ __forceinline__ int named_window_start(const int32_t *g, int64_t ld, int levels, int p) {
    const int d = g[p];
    int pos = p;  // the gaps [pos, p) are all deeper than d
    for (int l = levels - 1; l >= 0; --l)
        if (pos >= (1 << l) && g[l * ld + pos - (1 << l)] > d) pos -= 1 << l;
    return pos > 0 && g[pos - 1] == d ? -1 : pos;
}

// Last tip of the window of gap p: the tip before the nearest gap right of p shallower than g[p], or n.
__device__ __forceinline__ int window_end(const int32_t *g, int64_t ld, int levels, int n, int p) {
    const int d = g[p];
    int pos = p + 1;  // the gaps (p, pos) are all at least d deep
    for (int l = levels - 1; l >= 0; --l)
        if (pos + (1 << l) <= n && g[l * ld + pos] >= d) pos += 1 << l;
    return pos;
}

// The t' positions of tree t's tour restricted to the taxa of `bits`: flag[j] = t' position of tour position j (an
// exclusive scan of the kept flags) and kidx[p] = tour position of t' tip p.  Returns the number kept.
__device__ int restrict_tour(const PairArgs &a, int t, const uint32_t *bits, int32_t *flag, int32_t *kidx, int32_t *sums) {
    const int64_t lb = a.leaf_off[t];
    const int nl = static_cast<int>(a.leaf_off[t + 1] - lb);
    const int32_t *lt = a.leaf_taxon + lb;
    for (int j = threadIdx.x; j < nl; j += blockDim.x) {
        const int x = lt[j];
        flag[j] = (bits[x >> 5] >> (x & 31)) & 1u;
    }
    __syncthreads();
    const int k = block_scan(flag, nl, sums);
    for (int j = threadIdx.x; j < nl; j += blockDim.x)
        if ((j + 1 < nl ? flag[j + 1] : k) > flag[j]) kidx[flag[j]] = j;
    __syncthreads();
    return k;
}

// g[p] (level 0 of a gap table) for p in [0, k - 1): depth in t of the LCA of t' tips p and p + 1
__device__ void gap_depths(const PairArgs &a, int t, const int32_t *kidx, int k, int32_t *g) {
    const int64_t lb = a.leaf_off[t];
    for (int p = threadIdx.x; p + 1 < k; p += blockDim.x) {
        const int lo = kidx[p], hi = kidx[p + 1] - 1;  // adj_depth[j] is the LCA depth of tour positions j and j + 1
        const int l = 31 - __clz(hi - lo + 1);
        g[p] = min(a.tour_min[l * a.leaves + lb + lo], a.tour_min[l * a.leaves + lb + hi - (1 << l) + 1]);
    }
}

__global__ void __launch_bounds__(kThreads) pw_pairs(PairArgs a) {
    extern __shared__ uint32_t smem[];
    uint32_t *bits = smem;
    int32_t *wpre = reinterpret_cast<int32_t *>(smem + a.words);
    __shared__ int32_t sums[33];
    __shared__ int32_t tally[3];  // windows named in t_i', in t_j', windows of t_i' that are clusters of t_j'
    __shared__ long long item;
    const int64_t ld = a.max_k;
    int32_t *flag = a.scratch + blockIdx.x * a.slot;
    int32_t *kidx = flag + a.max_leaves + 1, *jpos = kidx + ld;
    int32_t *gi = jpos + ld, *gj = gi + a.levels * ld, *qlo = gj + a.levels * ld, *qhi = qlo + a.levels * ld;
    for (;;) {
        if (threadIdx.x == 0) item = static_cast<long long>(atomicAdd(a.next, 1ull));
        __syncthreads();
        const int64_t it = item;
        if (it >= a.pairs) return;
        // after the barrier above: thread 0 has read the previous pair's tallies; the barriers below order these
        // stores before the first atomicAdd
        if (threadIdx.x < 3) tally[threadIdx.x] = 0;
        const int ti = a.list[it].x, tj = a.list[it].y;
        const uint32_t *ri = a.bits + static_cast<int64_t>(ti) * a.words, *rj = a.bits + static_cast<int64_t>(tj) * a.words;
        for (int w = threadIdx.x; w < a.words; w += blockDim.x) {
            bits[w] = ri[w] & rj[w];
            wpre[w] = __popc(bits[w]);
        }
        __syncthreads();
        block_scan(wpre, a.words, sums);

        // t_j': rank in X -> t_j' position, and its gaps
        const int k = restrict_tour(a, tj, bits, flag, kidx, sums);
        {
            const int32_t *lt = a.leaf_taxon + a.leaf_off[tj];
            for (int q = threadIdx.x; q < k; q += blockDim.x) jpos[bitmap_rank(bits, wpre, lt[kidx[q]])] = q;
        }
        gap_depths(a, tj, kidx, k, gj);
        // t_i': the t_j' position of every t_i' tip, and its gaps
        restrict_tour(a, ti, bits, flag, kidx, sums);
        {
            const int32_t *lt = a.leaf_taxon + a.leaf_off[ti];
            for (int p = threadIdx.x; p < k; p += blockDim.x) qlo[p] = qhi[p] = jpos[bitmap_rank(bits, wpre, lt[kidx[p]])];
        }
        gap_depths(a, ti, kidx, k, gi);
        const int levels = 32 - __clz(k);  // 2^levels > k
        for (int l = 1; l < levels; ++l) {
            __syncthreads();
            const int half = 1 << (l - 1);
            const int64_t lo = (l - 1) * ld, hi = l * ld;
            for (int p = threadIdx.x; p + (1 << l) <= k; p += blockDim.x) {
                qlo[hi + p] = min(qlo[lo + p], qlo[lo + p + half]);
                qhi[hi + p] = max(qhi[lo + p], qhi[lo + p + half]);
                if (p + (1 << l) <= k - 1) {
                    gi[hi + p] = min(gi[lo + p], gi[lo + p + half]);
                    gj[hi + p] = min(gj[lo + p], gj[lo + p + half]);
                }
            }
        }
        __syncthreads();

        int named_i = 0, named_j = 0, both = 0;
        const int gaps = k - 1;
        for (int p = threadIdx.x; p < gaps; p += blockDim.x) {
            named_j += named_window_start(gj, ld, levels, p) >= 0;
            const int l = named_window_start(gi, ld, levels, p);
            if (l < 0) continue;
            ++named_i;
            const int r = window_end(gi, ld, levels, gaps, p);
            if (l == 0 && r == gaps) continue;  // X itself
            const int lo = table_min(qlo, ld, l, r), hi = table_max(qhi, ld, l, r);
            if (hi - lo != r - l) continue;
            const int d = table_min(gj, ld, lo, hi - 1);
            both += (lo == 0 || gj[lo - 1] < d) && (hi == gaps || gj[hi] < d);
        }
        if (named_i) atomicAdd(&tally[0], named_i);
        if (named_j) atomicAdd(&tally[1], named_j);
        if (both) atomicAdd(&tally[2], both);
        __syncthreads();
        if (threadIdx.x == 0) {  // the root window is named once in each tree
            a.clusters[static_cast<int64_t>(ti) * a.T + tj] = tally[0] - 1;
            a.clusters[static_cast<int64_t>(tj) * a.T + ti] = tally[1] - 1;
            a.common[static_cast<int64_t>(ti) * a.T + tj] = tally[2];
            a.common[static_cast<int64_t>(tj) * a.T + ti] = tally[2];
        }
    }
}

}  // namespace
}  // namespace scs

using namespace scs;

extern "C" int scs_forest_pairwise_rf(scs_ctx *ctx, const scs_forest *forest, int32_t *shared_taxa, int32_t *clusters,
                                      int32_t *common) {
    if (!ctx) return SCS_ERR_INVALID;
    if (!forest || !shared_taxa || !clusters || !common) return fail(ctx, SCS_ERR_INVALID, "scs_forest_pairwise_rf: bad argument");
    const int T = forest->num_trees(), taxa = forest->num_taxa;
    const int words = std::max(1, ceil_div(taxa, 32));
    const size_t smem = static_cast<size_t>(words) * 8;
    if (smem + 1024 > ctx->smem_optin)  // room for the static shared arrays
        return fail(ctx, SCS_ERR_INVALID, "scs_forest_pairwise_rf: too many taxa for the shared-memory bitmap of a pair");
    const int64_t nb = (static_cast<int64_t>(T) + kTile - 1) / kTile, tiles = nb * (nb + 1) / 2;
    if (tiles > INT_MAX)
        return fail(ctx, SCS_ERR_INVALID, "scs_forest_pairwise_rf: too many trees for the grid of pair tiles");
    if (T == 0) return SCS_OK;
    const size_t TT = static_cast<size_t>(T) * static_cast<size_t>(T);
    const std::vector<int64_t> &loff = forest->leaf_offsets;
    int64_t max_leaves = 0;
    for (int t = 0; t < T; ++t) max_leaves = std::max(max_leaves, loff[t + 1] - loff[t]);

    DevForest df;
    DevTours tours;
    GrowBuf ident, flags, bits, d_shared, d_clusters, d_common, list, counters, table, scratch;
    auto cleanup = [&] {
        df.free_all(ctx);
        tours.free_all(ctx);
        for (GrowBuf *b : {&ident, &flags, &bits, &d_shared, &d_clusters, &d_common, &list, &counters, &table, &scratch})
            release(ctx, *b);
        cudaStreamSynchronize(ctx->stream);
    };
    auto run = [&]() -> int {
        int rc;
        if ((rc = devforest_upload(ctx, forest, 0, &df))) return rc;
        const size_t words_bytes = static_cast<size_t>(T) * words * sizeof(uint32_t);
        const size_t list_bytes = (static_cast<size_t>(T) * (T + 1) / 2) * sizeof(int2);
        if ((rc = grow(ctx, bits, words_bytes)) || (rc = grow(ctx, d_shared, TT * 4)) || (rc = grow(ctx, d_clusters, TT * 4)) ||
            (rc = grow(ctx, d_common, TT * 4)) || (rc = grow(ctx, list, list_bytes)) || (rc = grow(ctx, counters, 24)))
            return rc;
        SCS_CUDA(ctx, cudaMemsetAsync(bits.ptr, 0, words_bytes, ctx->stream));
        SCS_CUDA(ctx, cudaMemsetAsync(d_clusters.ptr, 0, TT * 4, ctx->stream));
        SCS_CUDA(ctx, cudaMemsetAsync(d_common.ptr, 0, TT * 4, ctx->stream));
        SCS_CUDA(ctx, cudaMemsetAsync(counters.ptr, 0, 24, ctx->stream));
        unsigned long long *count = counters.as<unsigned long long>();  // listed pairs, largest k, next pair of pass 2
        int *max_k = reinterpret_cast<int *>(count + 1);

        // pass 1: bitmaps, shared taxa of every pair, the work list
        pw_bitmap<<<T, kThreads, 0, ctx->stream>>>(df.tree_off.as<int64_t>(), df.taxon.as<int32_t>(), taxa, words,
                                                   bits.as<uint32_t>());
        SCS_LAUNCHED(ctx, "pw_bitmap");
        pw_shared<<<static_cast<int>(tiles), kThreads, 0, ctx->stream>>>(T, words, bits.as<uint32_t>(), d_shared.as<int32_t>(),
                                                                         list.as<int2>(), count, max_k);
        SCS_LAUNCHED(ctx, "pw_shared");
        struct {
            unsigned long long pairs;
            int32_t max_k, pad;
        } head{};
        SCS_CUDA(ctx, cudaMemcpyAsync(&head, counters.ptr, 16, cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));

        if (head.pairs > 0) {
            // pass 2: tours, their sparse table, one CTA per listed pair
            std::vector<int32_t> identity(static_cast<size_t>(taxa > 0 ? taxa : 1));
            for (size_t x = 0; x < identity.size(); ++x) identity[x] = static_cast<int32_t>(x);
            if ((rc = grow(ctx, ident, identity.size() * sizeof(int32_t))) || (rc = grow(ctx, flags, 2 * sizeof(int32_t))))
                return rc;
            SCS_CUDA(ctx, cudaMemcpyAsync(ident.ptr, identity.data(), identity.size() * sizeof(int32_t), cudaMemcpyHostToDevice,
                                          ctx->stream));
            SCS_CUDA(ctx, cudaMemsetAsync(flags.ptr, 0, 2 * sizeof(int32_t), ctx->stream));
            if ((rc = devforest_tours(ctx, df, 0, ident.as<int32_t>(), &tours, flags.as<int32_t>()))) return rc;
            const int64_t leaves = df.leaves;
            int tour_levels = 1;
            while ((int64_t(1) << tour_levels) <= max_leaves) ++tour_levels;
            if ((rc = grow(ctx, table, static_cast<size_t>(leaves) * tour_levels * sizeof(int32_t)))) return rc;
            SCS_CUDA(ctx, cudaMemcpyAsync(table.ptr, tours.adj_depth.ptr, static_cast<size_t>(leaves) * sizeof(int32_t),
                                          cudaMemcpyDeviceToDevice, ctx->stream));
            pw_tour_table<<<T, kThreads, 0, ctx->stream>>>(df.leaf_off.as<int64_t>(), leaves, table.as<int32_t>());
            SCS_LAUNCHED(ctx, "pw_tour_table");

            const int64_t mk = head.max_k;
            int levels = 1;
            while ((int64_t(1) << levels) <= mk) ++levels;
            const int64_t slot = (max_leaves + 1) + 2 * mk + 4 * static_cast<int64_t>(levels) * mk;
            if (smem > 48 * 1024)
                SCS_CUDA(ctx, cudaFuncSetAttribute(pw_pairs, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
            int per_sm = 0;
            SCS_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pw_pairs, kThreads, smem));
            int64_t ctas = static_cast<int64_t>(std::max(per_sm, 1)) * ctx->sm_count;
            ctas = std::min<int64_t>(ctas, std::max<int64_t>(1, static_cast<int64_t>(kScratchBytes / (slot * sizeof(int32_t)))));
            ctas = std::min<int64_t>(ctas, static_cast<int64_t>(head.pairs));
            if ((rc = grow(ctx, scratch, static_cast<size_t>(ctas * slot) * sizeof(int32_t)))) return rc;

            PairArgs args{};
            args.T = T;
            args.words = words;
            args.bits = bits.as<uint32_t>();
            args.leaf_off = df.leaf_off.as<int64_t>();
            args.leaf_taxon = tours.leaf_taxon.as<int32_t>();
            args.tour_min = table.as<int32_t>();
            args.leaves = leaves;
            args.list = list.as<int2>();
            args.pairs = static_cast<int64_t>(head.pairs);
            args.next = count + 2;
            args.scratch = scratch.as<int32_t>();
            args.slot = slot;
            args.max_leaves = max_leaves;
            args.max_k = mk;
            args.levels = levels;
            args.clusters = d_clusters.as<int32_t>();
            args.common = d_common.as<int32_t>();
            pw_pairs<<<static_cast<int>(ctas), kThreads, smem, ctx->stream>>>(args);
            SCS_LAUNCHED(ctx, "pw_pairs");
        }
        SCS_CUDA(ctx, cudaMemcpyAsync(shared_taxa, d_shared.ptr, TT * 4, cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaMemcpyAsync(clusters, d_clusters.ptr, TT * 4, cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaMemcpyAsync(common, d_common.ptr, TT * 4, cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        ctx->d2h_bytes += static_cast<int64_t>(3 * TT * 4 + 16);
        return SCS_OK;
    };
    const int rc = run();
    cleanup();
    return rc;
}
