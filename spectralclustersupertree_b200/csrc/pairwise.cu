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
//
// Rooted triplet distances (scs_forest_pairwise_triplets) share pass 1 (PairPass).  Pass 2 (pw_triplets) is the row
// pass of triplets.cu with the supertree replaced by t_j: per row a of t_i', alpha comes from the gaps of t_i' and
// beta(x) = depth in t_j of LCA(a, x) from one range minimum of t_j's unrestricted tour, counted with a Fenwick tree
// and histogram over beta (dominance.cuh).  Work items are chunks of a pair's rows, so one large pair spreads over
// many CTAs; the row sums go to per-pair int64 accumulators with integer atomics, which pw_triplet_out halves into
// both triangles.

#include <algorithm>
#include <climits>
#include <string>
#include <vector>

#include "devforest.cuh"
#include "dominance.cuh"
#include "forest.hpp"
#include "supertree.cuh"

namespace scs {
namespace {

constexpr int kThreads = 256;
constexpr int kTile = 64;       // trees per side of a pass-1 tile (16 x 16 threads, 4 x 4 pairs each)
constexpr int kTileWords = 32;  // bitmap words per pass-1 stage
constexpr size_t kScratchBytes = size_t(4096) << 20;  // per-CTA scratch of pass 2, all resident CTAs together
constexpr int kRowWarps = kThreads / 32;  // row warps of a pw_triplets CTA when the trees are shallow enough
constexpr int kChunkRows = 512;           // rows of a pair one pw_triplets work item counts

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
    // pw_triplets: k of every pair; log2 of the row chunks per listed pair, ints per shared-memory array of a row warp
    // and row warps per CTA; the doubled row sums of every listed pair ([pairs][4]) and the T x T results
    const int32_t *shared;
    int32_t chunk_bits, stride, warps;
    unsigned long long *acc;
    int64_t *resolved, *agree, *contradict;
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

// Depth in t of the LCA of the tips at tour positions p != q of tree t (its tour's table at tab = tour_min + leaf_off[t])
__device__ __forceinline__ int tour_lca_depth(const int32_t *tab, int64_t ld, int p, int q) {
    const int lo = min(p, q), hi = max(p, q) - 1;  // adj_depth[j] is the LCA depth of tour positions j and j + 1
    const int l = 31 - __clz(hi - lo + 1);
    return min(__ldg(tab + l * ld + lo), __ldg(tab + l * ld + hi - (1 << l) + 1));
}

// Row a = t_i' position qa of a pair, one warp (the triplet row of triplets.cu with S = t_j): alpha(x) = depth in t_i
// of LCA(a, x) grows out of the gaps td of t_i', beta(x) = depth in t_j of LCA(a, x) is one range minimum over t_j's
// unrestricted tour between the tour positions jp of a and x.  Every beta is at most one of the two gap depths beside
// a in t_j's tour, so the Fenwick tree over beta + 1 in [1, m] and the histogram of beta in [0, m) take m + 1 ints
// each, m = 1 + the larger of those.  Adds to the lane's partial sums of the four doubled counts, except for the
// C(k - 1, 2) pairs of the row that r2 starts from.
__device__ __forceinline__ void pair_row(const PairArgs &a, const int32_t *tabj, int nlj, const int32_t *td,
                                         const int32_t *jp, int k, int qa, int lane, int32_t *fw, int32_t *hist,
                                         long long &r1, long long &r2, long long &ag, long long &co) {
    const int pa = jp[qa];
    const int m = 1 + max(pa > 0 ? tabj[pa - 1] : -1, pa + 1 < nlj ? tabj[pa] : -1);
    for (int i = lane; i <= m; i += 32) fw[i] = 0;
    for (int i = lane; i < m; i += 32) hist[i] = 0;
    __syncwarp();
    int L = qa, R = qa, inside = 0;  // t_i' positions [L, R] are inside the window (a itself is no point)
    for (;;) {
        int nL, nR;
        if (grow_window(td, k, lane, L, R, nL, nR) < 0) break;
        const int left = L - nL, added = left + nR - R;
        // the new taxa x (alpha(x) = level) against the y inside (alpha(y) > level): concordant when beta(y) >
        // beta(x), discordant when beta(y) < beta(x)
        for (int i = lane; i < added; i += 32) {
            const int b = tour_lca_depth(tabj, a.leaves, pa, jp[i < left ? nL + i : R + 1 + (i - left)]);
            const int below = fenwick_prefix(fw, b);
            co += below;
            ag += inside - below - hist[b];
        }
        __syncwarp();
        for (int i = lane; i < added; i += 32) {
            const int b = tour_lca_depth(tabj, a.leaves, pa, jp[i < left ? nL + i : R + 1 + (i - left)]);
            fenwick_add(fw, b + 1, m, 1);
            atomicAdd(&hist[b], 1);
        }
        __syncwarp();
        if (lane == 0) r1 += static_cast<long long>(inside) * added;
        inside += added;
        L = nL;
        R = nR;
    }
    // pairs {b, x} with beta(b) = beta(x), taken off the row's C(k - 1, 2) pairs by the caller
    for (int i = lane; i < m; i += 32) r2 -= static_cast<long long>(hist[i]) * (hist[i] - 1) / 2;
    __syncwarp();  // the next row clears the arrays
}

// Persistent CTAs taking work items from a counter: item it is rows [c * kChunkRows, (c + 1) * kChunkRows) of listed
// pair it >> chunk_bits, c = the low chunk_bits bits of it (none if that is past k).  X and its ranks as in pw_pairs; jtour[r] = position in
// t_j's unrestricted tour of the taxon of rank r; t_i's tour restricted to X gives, per t_i' position q, the t_j tour
// position jp[q] of its taxon and td[q], the depth in t_i of the LCA of t_i' positions q and q + 1.  The row warps
// then reuse the shared memory of the bitmap for their Fenwick trees and histograms; their sums go to the pair's
// accumulators as exact integer atomics, so the order in which CTAs take items changes no bit.
__global__ void __launch_bounds__(kThreads) pw_triplets(PairArgs a) {
    extern __shared__ uint32_t smem[];
    uint32_t *bits = smem;
    int32_t *wpre = reinterpret_cast<int32_t *>(smem + a.words);
    __shared__ int32_t sums[33];
    __shared__ long long item;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t ld = a.max_k;
    int32_t *flag = a.scratch + blockIdx.x * a.slot;
    int32_t *kidx = flag + a.max_leaves + 1, *jtour = kidx + ld, *jp = jtour + ld, *td = jp + ld;
    int32_t *fw = reinterpret_cast<int32_t *>(smem) + warp * 2 * a.stride, *hist = fw + a.stride;
    for (;;) {
        if (threadIdx.x == 0) item = static_cast<long long>(atomicAdd(a.next, 1ull));
        __syncthreads();
        const int64_t it = item;
        if (it >= a.pairs << a.chunk_bits) return;
        const int64_t pair = it >> a.chunk_bits;
        const int ti = a.list[pair].x, tj = a.list[pair].y;
        const int k = a.shared[static_cast<int64_t>(ti) * a.T + tj];
        const int row0 = static_cast<int>(it & ((int64_t(1) << a.chunk_bits) - 1)) * kChunkRows;
        if (row0 >= k) {  // past the pair's rows: every thread reads `item` before thread 0 takes the next one
            __syncthreads();
            continue;
        }
        const uint32_t *ri = a.bits + static_cast<int64_t>(ti) * a.words, *rj = a.bits + static_cast<int64_t>(tj) * a.words;
        for (int w = threadIdx.x; w < a.words; w += blockDim.x) {
            bits[w] = ri[w] & rj[w];
            wpre[w] = __popc(bits[w]);
        }
        __syncthreads();
        block_scan(wpre, a.words, sums);

        // t_j: rank in X -> unrestricted tour position
        const int64_t lbj = a.leaf_off[tj];
        const int nlj = static_cast<int>(a.leaf_off[tj + 1] - lbj);
        {
            const int32_t *lt = a.leaf_taxon + lbj;
            for (int j = threadIdx.x; j < nlj; j += blockDim.x) {
                const int x = lt[j];
                if ((bits[x >> 5] >> (x & 31)) & 1u) jtour[bitmap_rank(bits, wpre, x)] = j;
            }
        }
        // t_i': the t_j tour position of every t_i' tip, and its gaps (restrict_tour's barriers order jtour)
        restrict_tour(a, ti, bits, flag, kidx, sums);
        {
            const int32_t *lt = a.leaf_taxon + a.leaf_off[ti];
            for (int p = threadIdx.x; p < k; p += blockDim.x) jp[p] = jtour[bitmap_rank(bits, wpre, lt[kidx[p]])];
        }
        gap_depths(a, ti, kidx, k, td);
        __syncthreads();  // bits and wpre are free from here: the rows' Fenwick trees and histograms take their place

        if (warp < a.warps) {
            const int32_t *tabj = a.tour_min + lbj;
            const int row1 = min(k, row0 + kChunkRows);
            long long r1 = 0, r2 = 0, ag = 0, co = 0;
            int rows = 0;
            for (int qa = row0 + warp; qa < row1; qa += a.warps, ++rows)
                pair_row(a, tabj, nlj, td, jp, k, qa, lane, fw, hist, r1, r2, ag, co);
            if (lane == 0) r2 += static_cast<long long>(rows) * ((k - 1) * static_cast<long long>(k - 2) / 2);
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                r1 += __shfl_down_sync(0xffffffffu, r1, off);
                r2 += __shfl_down_sync(0xffffffffu, r2, off);
                ag += __shfl_down_sync(0xffffffffu, ag, off);
                co += __shfl_down_sync(0xffffffffu, co, off);
            }
            if (lane == 0) {
                unsigned long long *acc = a.acc + 4 * pair;
                if (r1) atomicAdd(acc, static_cast<unsigned long long>(r1));
                if (r2) atomicAdd(acc + 1, static_cast<unsigned long long>(r2));
                if (ag) atomicAdd(acc + 2, static_cast<unsigned long long>(ag));
                if (co) atomicAdd(acc + 3, static_cast<unsigned long long>(co));
            }
        }
        // the barrier at the top of the loop keeps the next item's bitmap out of the rows' arrays
    }
}

// One thread per listed pair (i, j): its doubled sums halved as tp_reduce halves them (a resolved or agreeing triplet
// is seen from two rows, a contradicting one from one) into both triangles; row i of `resolved` counts tree i.
__global__ void pw_triplet_out(PairArgs a) {
    const int64_t p = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (p >= a.pairs) return;
    const int64_t i = a.list[p].x, j = a.list[p].y;
    const unsigned long long *s = a.acc + 4 * p;
    a.resolved[i * a.T + j] = static_cast<int64_t>(s[0] / 2);
    a.resolved[j * a.T + i] = static_cast<int64_t>(s[1] / 2);
    a.agree[i * a.T + j] = a.agree[j * a.T + i] = static_cast<int64_t>(s[2] / 2);
    a.contradict[i * a.T + j] = a.contradict[j * a.T + i] = static_cast<int64_t>(s[3]);
}

// Pass 1 and what pass 2 of both entry points reads: the forest's taxon bitmaps, k of every pair, the work list of the
// pairs i <= j with k >= 3 and the largest such k; when the list is not empty, the forest's tours (weighting one) and
// the sparse table over them.
struct PairPass {
    int T = 0, taxa = 0, words = 0;
    size_t smem = 0;  // the bitmap of a pair and the prefix of its word popcounts in shared memory
    int64_t max_leaves = 0, pairs = 0, max_k = 0;
    DevForest df;
    DevTours tours;
    GrowBuf ident, flags, bits, d_shared, list, counters, table;

    // Host side: the limits of the bitmap and of the tile grid (failure status, message set, or SCS_OK).
    int prepare(scs_ctx *ctx, const char *name, const scs_forest *forest) {
        T = forest->num_trees();
        taxa = forest->num_taxa;
        words = std::max(1, ceil_div(taxa, 32));
        smem = static_cast<size_t>(words) * 8;
        if (smem + 1024 > ctx->smem_optin)  // room for the static shared arrays
            return fail(ctx, SCS_ERR_INVALID, (std::string(name) + ": too many taxa for the shared-memory bitmap of a pair").c_str());
        const int64_t nb = (static_cast<int64_t>(T) + kTile - 1) / kTile;
        if (nb * (nb + 1) / 2 > INT_MAX)
            return fail(ctx, SCS_ERR_INVALID, (std::string(name) + ": too many trees for the grid of pair tiles").c_str());
        const std::vector<int64_t> &loff = forest->leaf_offsets;
        for (int t = 0; t < T; ++t) max_leaves = std::max(max_leaves, loff[t + 1] - loff[t]);
        return SCS_OK;
    }

    // The device side (T > 0); returns after the work list's length and largest k are on the host.
    int run(scs_ctx *ctx, const scs_forest *forest) {
        int rc;
        if ((rc = devforest_upload(ctx, forest, 0, &df))) return rc;
        const size_t TT = static_cast<size_t>(T) * static_cast<size_t>(T);
        const size_t words_bytes = static_cast<size_t>(T) * words * sizeof(uint32_t);
        const size_t list_bytes = (static_cast<size_t>(T) * (T + 1) / 2) * sizeof(int2);
        if ((rc = grow(ctx, bits, words_bytes)) || (rc = grow(ctx, d_shared, TT * 4)) || (rc = grow(ctx, list, list_bytes)) ||
            (rc = grow(ctx, counters, 24)))
            return rc;
        SCS_CUDA(ctx, cudaMemsetAsync(bits.ptr, 0, words_bytes, ctx->stream));
        SCS_CUDA(ctx, cudaMemsetAsync(counters.ptr, 0, 24, ctx->stream));
        const int nb = (T + kTile - 1) / kTile;
        pw_bitmap<<<T, kThreads, 0, ctx->stream>>>(df.tree_off.as<int64_t>(), df.taxon.as<int32_t>(), taxa, words,
                                                   bits.as<uint32_t>());
        SCS_LAUNCHED(ctx, "pw_bitmap");
        pw_shared<<<nb * (nb + 1) / 2, kThreads, 0, ctx->stream>>>(T, words, bits.as<uint32_t>(), d_shared.as<int32_t>(),
                                                                   list.as<int2>(), count(), max_k_dev());
        SCS_LAUNCHED(ctx, "pw_shared");
        struct {
            unsigned long long pairs;
            int32_t max_k, pad;
        } head{};
        SCS_CUDA(ctx, cudaMemcpyAsync(&head, counters.ptr, 16, cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        pairs = static_cast<int64_t>(head.pairs);
        max_k = head.max_k;
        if (pairs == 0) return SCS_OK;
        std::vector<int32_t> identity(static_cast<size_t>(taxa > 0 ? taxa : 1));
        for (size_t x = 0; x < identity.size(); ++x) identity[x] = static_cast<int32_t>(x);
        if ((rc = grow(ctx, ident, identity.size() * sizeof(int32_t))) || (rc = grow(ctx, flags, 2 * sizeof(int32_t))))
            return rc;
        SCS_CUDA(ctx, cudaMemcpyAsync(ident.ptr, identity.data(), identity.size() * sizeof(int32_t), cudaMemcpyHostToDevice,
                                      ctx->stream));
        SCS_CUDA(ctx, cudaMemsetAsync(flags.ptr, 0, 2 * sizeof(int32_t), ctx->stream));
        if ((rc = devforest_tours(ctx, df, 0, ident.as<int32_t>(), &tours, flags.as<int32_t>()))) return rc;
        int tour_levels = 1;
        while ((int64_t(1) << tour_levels) <= max_leaves) ++tour_levels;
        if ((rc = grow(ctx, table, static_cast<size_t>(df.leaves) * tour_levels * sizeof(int32_t)))) return rc;
        SCS_CUDA(ctx, cudaMemcpyAsync(table.ptr, tours.adj_depth.ptr, static_cast<size_t>(df.leaves) * sizeof(int32_t),
                                      cudaMemcpyDeviceToDevice, ctx->stream));
        pw_tour_table<<<T, kThreads, 0, ctx->stream>>>(df.leaf_off.as<int64_t>(), df.leaves, table.as<int32_t>());
        SCS_LAUNCHED(ctx, "pw_tour_table");
        return SCS_OK;
    }

    // listed pairs, largest k, next item of pass 2
    unsigned long long *count() const { return counters.as<unsigned long long>(); }
    int *max_k_dev() const { return reinterpret_cast<int *>(count() + 1); }

    // The fields of pass 2's arguments that pass 1 gives.
    void fill(PairArgs *args) const {
        args->T = T;
        args->words = words;
        args->bits = bits.as<uint32_t>();
        args->leaf_off = df.leaf_off.as<int64_t>();
        args->leaf_taxon = tours.leaf_taxon.as<int32_t>();
        args->tour_min = table.as<int32_t>();
        args->leaves = df.leaves;
        args->list = list.as<int2>();
        args->pairs = pairs;
        args->next = count() + 2;
        args->max_leaves = max_leaves;
        args->max_k = max_k;
    }

    // Resident CTAs of a pass-2 kernel with `dyn` bytes of shared memory, at most `work` and at most what
    // kScratchBytes of per-CTA scratch of `slot` ints allows.
    template <typename K>
    int ctas(scs_ctx *ctx, K kernel, size_t dyn, int64_t slot, int64_t work, int64_t *out) const {
        if (dyn > 48 * 1024)
            SCS_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(dyn)));
        int per_sm = 0;
        SCS_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kThreads, dyn));
        int64_t n = static_cast<int64_t>(std::max(per_sm, 1)) * ctx->sm_count;
        n = std::min<int64_t>(n, std::max<int64_t>(1, static_cast<int64_t>(kScratchBytes / (slot * sizeof(int32_t)))));
        *out = std::min<int64_t>(n, work);
        return SCS_OK;
    }

    void release_all(scs_ctx *ctx) {
        df.free_all(ctx);
        tours.free_all(ctx);
        for (GrowBuf *b : {&ident, &flags, &bits, &d_shared, &list, &counters, &table}) release(ctx, *b);
    }
};

}  // namespace
}  // namespace scs

using namespace scs;

extern "C" int scs_forest_pairwise_rf(scs_ctx *ctx, const scs_forest *forest, int32_t *shared_taxa, int32_t *clusters,
                                      int32_t *common) {
    if (!ctx) return SCS_ERR_INVALID;
    if (!forest || !shared_taxa || !clusters || !common) return fail(ctx, SCS_ERR_INVALID, "scs_forest_pairwise_rf: bad argument");
    PairPass p;
    int rc = p.prepare(ctx, "scs_forest_pairwise_rf", forest);
    if (rc) return rc;
    const int T = p.T;
    if (T == 0) return SCS_OK;
    const size_t TT = static_cast<size_t>(T) * static_cast<size_t>(T);

    GrowBuf d_clusters, d_common, scratch;
    auto cleanup = [&] {
        p.release_all(ctx);
        for (GrowBuf *b : {&d_clusters, &d_common, &scratch}) release(ctx, *b);
        cudaStreamSynchronize(ctx->stream);
    };
    auto run = [&]() -> int {
        if ((rc = grow(ctx, d_clusters, TT * 4)) || (rc = grow(ctx, d_common, TT * 4))) return rc;
        SCS_CUDA(ctx, cudaMemsetAsync(d_clusters.ptr, 0, TT * 4, ctx->stream));
        SCS_CUDA(ctx, cudaMemsetAsync(d_common.ptr, 0, TT * 4, ctx->stream));
        // pass 1: bitmaps, shared taxa of every pair, the work list, the tours and their sparse table
        if ((rc = p.run(ctx, forest))) return rc;

        if (p.pairs > 0) {
            // pass 2: one CTA per listed pair
            const int64_t mk = p.max_k;
            int levels = 1;
            while ((int64_t(1) << levels) <= mk) ++levels;
            const int64_t slot = (p.max_leaves + 1) + 2 * mk + 4 * static_cast<int64_t>(levels) * mk;
            int64_t ctas = 0;
            if ((rc = p.ctas(ctx, pw_pairs, p.smem, slot, p.pairs, &ctas))) return rc;
            if ((rc = grow(ctx, scratch, static_cast<size_t>(ctas * slot) * sizeof(int32_t)))) return rc;

            PairArgs args{};
            p.fill(&args);
            args.scratch = scratch.as<int32_t>();
            args.slot = slot;
            args.levels = levels;
            args.clusters = d_clusters.as<int32_t>();
            args.common = d_common.as<int32_t>();
            pw_pairs<<<static_cast<int>(ctas), kThreads, p.smem, ctx->stream>>>(args);
            SCS_LAUNCHED(ctx, "pw_pairs");
        }
        SCS_CUDA(ctx, cudaMemcpyAsync(shared_taxa, p.d_shared.ptr, TT * 4, cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaMemcpyAsync(clusters, d_clusters.ptr, TT * 4, cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaMemcpyAsync(common, d_common.ptr, TT * 4, cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        ctx->d2h_bytes += static_cast<int64_t>(3 * TT * 4 + 16);
        return SCS_OK;
    };
    rc = run();
    cleanup();
    return rc;
}

extern "C" int scs_forest_pairwise_triplets(scs_ctx *ctx, const scs_forest *forest, int32_t *shared_taxa,
                                            int64_t *resolved, int64_t *agree, int64_t *contradict) {
    if (!ctx) return SCS_ERR_INVALID;
    if (!forest || !shared_taxa || !resolved || !agree || !contradict)
        return fail(ctx, SCS_ERR_INVALID, "scs_forest_pairwise_triplets: bad argument");
    PairPass p;
    int rc = p.prepare(ctx, "scs_forest_pairwise_triplets", forest);
    if (rc) return rc;
    const int T = p.T;
    // the deepest tip of the forest bounds every beta of a row: two arrays of (depth + 1) ints per row warp
    int max_depth = 0;
    {
        const std::vector<int64_t> &noff = forest->node_offsets;
#pragma omp parallel num_threads(scs_host_threads()) reduction(max : max_depth)
        {
            std::vector<int32_t> depth;
#pragma omp for schedule(dynamic, 16)
            for (int t = 0; t < T; ++t) {
                const int64_t b = noff[t], n = noff[t + 1] - b;
                depth.assign(static_cast<size_t>(n), 0);
                for (int64_t u = 1; u < n; ++u) {  // parent < child within a tree
                    depth[u] = depth[forest->parent[b + u]] + 1;
                    max_depth = std::max(max_depth, depth[u]);
                }
            }
        }
    }
    const int stride = max_depth + 1;
    const size_t warp_smem = 2 * static_cast<size_t>(stride) * sizeof(int32_t);
    const int warps = static_cast<int>(std::min<size_t>(kRowWarps, (ctx->smem_optin - 1024) / warp_smem));
    if (warps < 1)
        return fail(ctx, SCS_ERR_INVALID,
                    "scs_forest_pairwise_triplets: a source tree is too deep for the shared-memory Fenwick tree of a row");
    if (T == 0) return SCS_OK;
    const size_t TT = static_cast<size_t>(T) * static_cast<size_t>(T);

    GrowBuf d_resolved, d_agree, d_contradict, acc, scratch;
    auto cleanup = [&] {
        p.release_all(ctx);
        for (GrowBuf *b : {&d_resolved, &d_agree, &d_contradict, &acc, &scratch}) release(ctx, *b);
        cudaStreamSynchronize(ctx->stream);
    };
    auto run = [&]() -> int {
        const size_t mat = TT * sizeof(int64_t);
        if ((rc = grow(ctx, d_resolved, mat)) || (rc = grow(ctx, d_agree, mat)) || (rc = grow(ctx, d_contradict, mat)))
            return rc;
        SCS_CUDA(ctx, cudaMemsetAsync(d_resolved.ptr, 0, mat, ctx->stream));
        SCS_CUDA(ctx, cudaMemsetAsync(d_agree.ptr, 0, mat, ctx->stream));
        SCS_CUDA(ctx, cudaMemsetAsync(d_contradict.ptr, 0, mat, ctx->stream));
        if ((rc = p.run(ctx, forest))) return rc;

        if (p.pairs > 0) {
            // pass 2: persistent CTAs over chunks of rows of the listed pairs
            const int64_t mk = p.max_k;
            int chunk_bits = 0;  // a power of two of row chunks per pair covers the largest k
            while ((int64_t(kChunkRows) << chunk_bits) < mk) ++chunk_bits;
            const int64_t slot = (p.max_leaves + 1) + 4 * mk;
            const size_t dyn = std::max(p.smem, static_cast<size_t>(warps) * warp_smem);
            int64_t ctas = 0;
            if ((rc = p.ctas(ctx, pw_triplets, dyn, slot, p.pairs << chunk_bits, &ctas))) return rc;
            const size_t acc_bytes = static_cast<size_t>(p.pairs) * 4 * sizeof(unsigned long long);
            if ((rc = grow(ctx, scratch, static_cast<size_t>(ctas * slot) * sizeof(int32_t))) || (rc = grow(ctx, acc, acc_bytes)))
                return rc;
            SCS_CUDA(ctx, cudaMemsetAsync(acc.ptr, 0, acc_bytes, ctx->stream));

            PairArgs args{};
            p.fill(&args);
            args.scratch = scratch.as<int32_t>();
            args.slot = slot;
            args.shared = p.d_shared.as<int32_t>();
            args.chunk_bits = chunk_bits;
            args.stride = stride;
            args.warps = warps;
            args.acc = acc.as<unsigned long long>();
            args.resolved = d_resolved.as<int64_t>();
            args.agree = d_agree.as<int64_t>();
            args.contradict = d_contradict.as<int64_t>();
            pw_triplets<<<static_cast<int>(ctas), kThreads, dyn, ctx->stream>>>(args);
            SCS_LAUNCHED(ctx, "pw_triplets");
            pw_triplet_out<<<static_cast<int>(ceil_div(p.pairs, kThreads)), kThreads, 0, ctx->stream>>>(args);
            SCS_LAUNCHED(ctx, "pw_triplet_out");
        }
        SCS_CUDA(ctx, cudaMemcpyAsync(shared_taxa, p.d_shared.ptr, TT * 4, cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaMemcpyAsync(resolved, d_resolved.ptr, mat, cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaMemcpyAsync(agree, d_agree.ptr, mat, cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaMemcpyAsync(contradict, d_contradict.ptr, mat, cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        ctx->d2h_bytes += static_cast<int64_t>(TT * 4 + 3 * mat + 16);
        return SCS_OK;
    };
    rc = run();
    cleanup();
    return rc;
}
