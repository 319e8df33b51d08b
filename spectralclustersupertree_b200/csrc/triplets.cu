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
//
// Per taxon (scs_supertree_taxon_triplets).  Each triplet is also credited to its three taxa.  For a point x of row a
// let f_alpha(x) / f_beta(x) be the other points y whose alpha / beta differs from x's, and c(x) / d(x) those with
// (alpha(x) - alpha(y)) (beta(x) - beta(y)) > 0 / < 0.  With R_p the sums over the points of row p and C_p the sums of
// the values of point p over the other rows of the tree, taxon p has (R_p[f_alpha] / 2 + C_p[f_alpha]) / 2 resolved
// source triplets, likewise with f_beta resolved supertree triplets and with c agreeing ones, and R_p[d] / 2 + C_p[d]
// contradicting ones: a resolved or agreeing triplet ab|x is seen from rows a and b and each of its taxa collects it
// twice (as the row or as one of its pair), a contradicting one is seen from one row and each taxon collects it once.
// The row warp regrows the window, now with every point's beta known in advance (a histogram over the row), and
// adds each point's four values into the column of its t' position; the columns go to a [chunk trees x taxa] matrix,
// which a last kernel adds up per taxon in tree order.
//
// MRP score (scs_supertree_mrp).  Every non-trivial cluster c of t' is a binary character (1 on c, 0 on X_t \ c,
// missing elsewhere) whose Fitch/Hartigan length on S equals its length on s' (a missing tip changes neither cost nor
// set at its parent).  The clusters of t' are the windows of t' positions around a gap q that hold every gap with
// td >= td[q]; gap q names its window's cluster when no gap left of it in the window has the same depth.  s' is the
// same kind of order: the shared taxa by S leaf position (S-rank r, from a bitmap over S's leaves) and sdep[r] = depth
// in S of the LCA of ranks r and r + 1.  Write x / y for the children of a node whose set is {0} / {1}: Hartigan's
// cost m - max(n_0, n_1) is min(x, y) and the set follows the sign of x - y, so a node needs only that difference
// (its balance), and a child adds one to the cost when it moves the balance towards 0.  Let w be the LCA in s' of the
// character's taxa: its ancestors each have one child holding the character and the rest all 0, so together with
// the all-0 outgroup they add 1 exactly when w's set is {1}.  One warp per gap finds the cluster and w's leaf range
// [lw, rw] with ballots, and one lane runs the stack-based Hartigan pass over that range, the ranks streamed in 32 at
// a time.  The stack holds (depth, balance) of the open nodes, at most one per level of S, in shared memory: the same
// two ints per level as the per-tree triplet row.  A character costs O(rw - lw + 1): |c| when S agrees with it, k at
// worst.

#include <algorithm>
#include <climits>
#include <string>
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
constexpr size_t kMatrixBytes = size_t(256) << 20;           // per-taxon counts of one chunk's trees

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
    int64_t *rows;   // per tree: [chunk leaves][4]: per row a: R1, R2, AG, CO; per taxon: [4][chunk leaves]: the
                     // columns of f_alpha, f_beta, c, d at each tree's t' positions, with R / 2 added at the row's own
    int64_t *per_tree;
    // per taxon
    const int32_t *s_taxon;  // S leaf position -> taxon
    const double *weight;    // [trees]
    int64_t *matrix;         // [chunk trees][4][taxa]: the four counts of every taxon in X_t, -1 for the others
    int64_t *per_taxon;      // [taxa][6]: trees, triplets, resolved source, resolved supertree, agree, contradict
    double *weighted;        // [taxa][3]: resolved source, agree, contradict summed with the tree weights
    // MRP score, per tree at its first tour position (in the scratch of `rows`)
    int32_t words;           // 32-bit words of a bitmap over S's leaf positions
    int32_t *sq;             // [chunk leaves]: t' position of the shared taxon of S-rank r
    int32_t *sr;             // [chunk leaves]: S-rank of t' position q
    int32_t *sdep;           // [chunk leaves]: depth in S of the LCA of S-ranks r and r + 1
    int32_t *len;            // [chunk leaves]: length of the character of gap q, 0 if gap q names no character
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

// The tree of chunk tour position g: the last t with leaf_off[t] <= leaf0 + g.
__device__ __forceinline__ int tree_of(const TripletArgs &a, int64_t g) {
    int lo = a.t0, hi = a.t1;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (a.leaf_off[mid] <= a.leaf0 + g) lo = mid; else hi = mid;
    }
    return lo;
}

// The next depth level of the window [L, R] of t' positions around a (-1 once the window is the whole tree), and the
// window [nL, nR] grown by it: its new positions are the taxa x with alpha(x) = level.  Called by the whole warp.
__device__ __forceinline__ int grow_window(const int32_t *td, int k, int lane, int L, int R, int &nL, int &nR) {
    const int eL = L > 0 ? td[L - 1] : -1, eR = R < k - 1 ? td[R] : -1;
    const int level = max(eL, eR);
    nL = L;
    nR = R;
    if (level < 0) return level;
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
    return level;
}

// Fenwick tree over [1, m] in shared memory: the sum of entries [1, f], and v added at f.
__device__ __forceinline__ int fenwick_prefix(const int32_t *fw, int f) {
    int s = 0;
    for (; f > 0; f -= f & -f) s += fw[f];
    return s;
}
__device__ __forceinline__ void fenwick_add(int32_t *fw, int f, int m, int v) {
    for (; f <= m; f += f & -f) atomicAdd(&fw[f], v);
}

// One warp per row: tour position g of the chunk.  Shared memory per warp: Fenwick tree over beta + 1 in [1, m] and
// a histogram of beta in [0, m), m = depth of a in S (beta < m).
__global__ void __launch_bounds__(kMaxRowWarps * 32, 1) tp_rows(TripletArgs a, int stride) {
    extern __shared__ int32_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t g = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + warp;
    if (g >= a.chunk_leaves) return;
    int64_t *out = a.rows + 4 * g;
    const int lo = tree_of(a, g);
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
        int nL, nR;
        if (grow_window(td, k, lane, L, R, nL, nR) < 0) break;
        const int left = L - nL, added = left + nR - R;
        // the new taxa x (alpha(x) = level) against the y inside (alpha(y) > level): concordant when beta(y) >
        // beta(x), discordant when beta(y) < beta(x)
        for (int i = lane; i < added; i += 32) {
            const int b = s_lca_depth(a, pa, sp[i < left ? nL + i : R + 1 + (i - left)]);
            const int below = fenwick_prefix(fw, b);
            co += below;
            ag += inside - below - hist[b];
        }
        __syncwarp();
        for (int i = lane; i < added; i += 32) {
            const int b = s_lca_depth(a, pa, sp[i < left ? nL + i : R + 1 + (i - left)]);
            fenwick_add(fw, b + 1, m, 1);
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

// One warp per row, for the per-taxon counts.  Every point x gets f_alpha(x), f_beta(x), c(x), d(x) (see the top of
// the file), added to the column of its t' position; half the row's sums go to the column of a.  Shared memory per
// warp, three arrays over [0, m]: lt[b] = points with beta < b (from a histogram of the whole row), a Fenwick tree
// over beta + 1 of the points inside the window (deeper in t than the level being added) and one of that level.
__global__ void __launch_bounds__(kMaxRowWarps * 32, 1) tx_rows(TripletArgs a, int stride) {
    extern __shared__ int32_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t g = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + warp;
    if (g >= a.chunk_leaves) return;
    const int lo = tree_of(a, g);
    const int64_t rel = a.leaf_off[lo] - a.leaf0;
    const int nl = static_cast<int>(a.leaf_off[lo + 1] - a.leaf_off[lo]), j = static_cast<int>(g - rel);
    const int k = a.k[lo - a.t0];
    const int32_t *qp = a.qpos + rel;
    const int qa = qp[j];
    if (k < 3 || (j + 1 < nl ? qp[j + 1] : k) == qa) return;  // fewer than three shared taxa, or a is not shared
    const int32_t *sp = a.spos + rel, *td = a.td + rel;
    const int pa = sp[qa], m = a.leaf_depth[pa];
    int32_t *lt = smem + warp * 3 * stride, *deep = lt + stride, *lev = deep + stride;
    for (int i = lane; i <= m; i += 32) lt[i] = deep[i] = lev[i] = 0;
    __syncwarp();
    for (int q = lane; q < k; q += 32)
        if (q != qa) atomicAdd(&lt[s_lca_depth(a, pa, sp[q]) + 1], 1);
    __syncwarp();
    for (int base = 0, carry = 0; base <= m; base += 32) {  // inclusive scan of the shifted histogram
        const int i = base + lane;
        int v = i <= m ? lt[i] : 0;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const int o = __shfl_up_sync(0xffffffffu, v, off);
            if (lane >= off) v += o;
        }
        if (i <= m) lt[i] = carry + v;
        carry += __shfl_sync(0xffffffffu, v, 31);
    }
    __syncwarp();

    unsigned long long *col = reinterpret_cast<unsigned long long *>(a.rows) + rel;
    const int64_t cs = a.chunk_leaves;
    long long s_fa = 0, s_fb = 0, s_c = 0, s_d = 0;
    int L = qa, R = qa, inside = 0;
    for (;;) {
        int nL, nR;
        if (grow_window(td, k, lane, L, R, nL, nR) < 0) break;
        const int left = L - nL, added = left + nR - R;
        auto point = [&](int i) { return i < left ? nL + i : R + 1 + (i - left); };
        for (int i = lane; i < added; i += 32) fenwick_add(lev, s_lca_depth(a, pa, sp[point(i)]) + 1, m, 1);
        __syncwarp();
        for (int i = lane; i < added; i += 32) {
            const int q = point(i), b = s_lca_depth(a, pa, sp[q]);
            // the other points with beta below / above x's: all of them, those inside (deeper), those of the level
            const int lt_all = lt[b], gt_all = k - 1 - lt[b + 1];
            const int lt_in = fenwick_prefix(deep, b), gt_in = inside - fenwick_prefix(deep, b + 1);
            const int lt_lv = fenwick_prefix(lev, b), gt_lv = added - fenwick_prefix(lev, b + 1);
            const int fa = k - 1 - added, fb = k - 1 - (lt[b + 1] - lt[b]);
            const int c = gt_in + (lt_all - lt_in - lt_lv);  // deeper with beta above, shallower with beta below
            const int d = lt_in + (gt_all - gt_in - gt_lv);  // deeper with beta below, shallower with beta above
            atomicAdd(col + q, static_cast<unsigned long long>(fa));
            atomicAdd(col + cs + q, static_cast<unsigned long long>(fb));
            atomicAdd(col + 2 * cs + q, static_cast<unsigned long long>(c));
            atomicAdd(col + 3 * cs + q, static_cast<unsigned long long>(d));
            s_fa += fa;
            s_fb += fb;
            s_c += c;
            s_d += d;
        }
        __syncwarp();
        for (int i = lane; i < added; i += 32) {
            const int f = s_lca_depth(a, pa, sp[point(i)]) + 1;
            fenwick_add(lev, f, m, -1);
            fenwick_add(deep, f, m, 1);
        }
        __syncwarp();
        inside += added;
        L = nL;
        R = nR;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        s_fa += __shfl_down_sync(0xffffffffu, s_fa, off);
        s_fb += __shfl_down_sync(0xffffffffu, s_fb, off);
        s_c += __shfl_down_sync(0xffffffffu, s_c, off);
        s_d += __shfl_down_sync(0xffffffffu, s_d, off);
    }
    if (lane == 0) {  // every pair of points is in the sums twice
        atomicAdd(col + qa, static_cast<unsigned long long>(s_fa / 2));
        atomicAdd(col + cs + qa, static_cast<unsigned long long>(s_fb / 2));
        atomicAdd(col + 2 * cs + qa, static_cast<unsigned long long>(s_c / 2));
        atomicAdd(col + 3 * cs + qa, static_cast<unsigned long long>(s_d / 2));
    }
}

// One warp per tree of the chunk with at least three shared taxa: its columns as the four counts of each of its taxa,
// into the tree's rows of the matrix.
__global__ void tx_tree(TripletArgs a) {
    const int64_t w = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= a.t1 - a.t0) return;
    const int k = a.k[w];
    if (k < 3) return;
    const int64_t rel = a.leaf_off[a.t0 + w] - a.leaf0, cs = a.chunk_leaves, taxa = a.taxa;
    const int64_t *col = a.rows + rel;
    const int32_t *sp = a.spos + rel;
    int64_t *out = a.matrix + w * 4 * taxa;
    for (int q = lane; q < k; q += 32) {
        const int x = a.s_taxon[sp[q]];
        out[x] = col[q] / 2;                       // resolved in t'
        out[taxa + x] = col[cs + q] / 2;           // resolved in s'
        out[2 * taxa + x] = col[2 * cs + q] / 2;   // agree
        out[3 * taxa + x] = col[3 * cs + q];       // contradict
    }
}

// One thread per taxon: the chunk's trees in order added to its counts, and to its weighted sums as acc + w * count
// without contraction, so the sums are those of the same loop on the host.
__global__ void tx_reduce(TripletArgs a) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= a.taxa) return;
    const int64_t taxa = a.taxa;
    int64_t *cnt = a.per_taxon + 6 * static_cast<int64_t>(x);
    double *sum = a.weighted + 3 * static_cast<int64_t>(x);
    long long c[6] = {cnt[0], cnt[1], cnt[2], cnt[3], cnt[4], cnt[5]};
    double s[3] = {sum[0], sum[1], sum[2]};
    for (int w = 0; w < a.t1 - a.t0; ++w) {
        const int64_t *m = a.matrix + w * 4 * taxa + x;
        const long long rs = m[0];
        if (rs < 0) continue;  // x is not in X_t, or k < 3
        const long long k = a.k[w], ag = m[2 * taxa], co = m[3 * taxa];
        const double wt = a.weight[a.t0 + w];
        c[0] += 1;
        c[1] += (k - 1) * (k - 2) / 2;
        c[2] += rs;
        c[3] += m[taxa];
        c[4] += ag;
        c[5] += co;
        s[0] = __dadd_rn(s[0], __dmul_rn(wt, static_cast<double>(rs)));
        s[1] = __dadd_rn(s[1], __dmul_rn(wt, static_cast<double>(ag)));
        s[2] = __dadd_rn(s[2], __dmul_rn(wt, static_cast<double>(co)));
    }
    for (int f = 0; f < 6; ++f) cnt[f] = c[f];
    for (int f = 0; f < 3; ++f) sum[f] = s[f];
}

// One CTA per tree with at least three shared taxa: S-ranks of its taxa and the depths between S-rank neighbours.
// Shared memory: a bitmap over S's leaf positions and the exclusive prefix of its word popcounts.
__global__ void __launch_bounds__(kPrepThreads) mp_rank(TripletArgs a) {
    extern __shared__ uint32_t bits[];
    int32_t *wpre = reinterpret_cast<int32_t *>(bits + a.words);
    __shared__ int32_t sums[33];
    const int w = blockIdx.x;
    const int k = a.k[w];
    if (k < 3) return;
    const int64_t rel = a.leaf_off[a.t0 + w] - a.leaf0;
    const int32_t *sp = a.spos + rel;
    int32_t *sq = a.sq + rel, *sr = a.sr + rel, *sd = a.sdep + rel;
    for (int i = threadIdx.x; i < a.words; i += blockDim.x) bits[i] = 0;
    __syncthreads();
    for (int q = threadIdx.x; q < k; q += blockDim.x) atomicOr(&bits[sp[q] >> 5], 1u << (sp[q] & 31));
    __syncthreads();
    for (int i = threadIdx.x; i < a.words; i += blockDim.x) wpre[i] = __popc(bits[i]);
    __syncthreads();
    block_scan(wpre, a.words, sums);
    for (int q = threadIdx.x; q < k; q += blockDim.x) {
        const int r = bitmap_rank(bits, wpre, sp[q]);
        sq[r] = q;
        sr[q] = r;
    }
    __syncthreads();
    for (int r = threadIdx.x; r < k - 1; r += blockDim.x) sd[r] = s_lca_depth(a, sp[sq[r]], sp[sq[r + 1]]);
}

// Hartigan: child of sign s (+1 set {0}, -1 set {1}, 0 set {0, 1}) added to a node of balance bal; returns the cost.
__device__ __forceinline__ int mp_attach(int &bal, int s) {
    const int cost = (s > 0 && bal < 0) || (s < 0 && bal > 0);
    bal += s;
    return cost;
}

// One warp per tour position of the chunk, for the gap q between t' positions q and q + 1 of its taxon: the length
// of the character that gap names, or 0.  Shared memory per warp: the stack of (depth, balance) of `stride` levels.
__global__ void __launch_bounds__(kMaxRowWarps * 32, 1) mp_chars(TripletArgs a, int stride) {
    extern __shared__ int32_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t g = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + warp;
    if (g >= a.chunk_leaves) return;
    const int lo_t = tree_of(a, g);
    const int64_t rel = a.leaf_off[lo_t] - a.leaf0;
    const int nl = static_cast<int>(a.leaf_off[lo_t + 1] - a.leaf_off[lo_t]), j = static_cast<int>(g - rel);
    const int k = a.k[lo_t - a.t0];
    const int32_t *qp = a.qpos + rel;
    const int q = qp[j];
    if (k < 3 || (j + 1 < nl ? qp[j + 1] : k) == q || q >= k - 1) return;  // no gap of a tree with characters
    const int32_t *td = a.td + rel, *sq = a.sq + rel, *sr = a.sr + rel, *sd = a.sdep + rel;
    int32_t *len = a.len + rel;
    const unsigned full = 0xffffffffu;
    const int d = td[q];
    // the cluster: t' positions [lo, hi] around gap q with every gap inside at depth >= d
    int lo = q;
    for (;;) {
        const int i = lo - 1 - lane;
        const unsigned stop = __ballot_sync(full, i < 0 || td[i] <= d);
        if (!stop) {
            lo -= 32;
            continue;
        }
        const int i0 = lo - __ffs(stop);
        if (i0 >= 0 && td[i0] == d) {  // an earlier gap of the same node names it
            if (lane == 0) len[q] = 0;
            return;
        }
        lo = i0 + 1;
        break;
    }
    int hi = q + 1;
    for (;;) {
        const int i = hi + lane;
        const unsigned stop = __ballot_sync(full, i >= k - 1 || td[i] < d);
        if (stop) {
            hi += __ffs(stop) - 1;
            break;
        }
        hi += 32;
    }
    if (lo == 0 && hi == k - 1) {  // X_t itself
        if (lane == 0) len[q] = 0;
        return;
    }
    // the S-ranks of the character's taxa, and w = their LCA in s': its depth dw and leaf range [lw, rw]
    int rmin = INT_MAX, rmax = -1;
    for (int i = lo + lane; i <= hi; i += 32) {
        const int r = sr[i];
        rmin = min(rmin, r);
        rmax = max(rmax, r);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        rmin = min(rmin, __shfl_xor_sync(full, rmin, off));
        rmax = max(rmax, __shfl_xor_sync(full, rmax, off));
    }
    int dw = INT_MAX;
    for (int r = rmin + lane; r < rmax; r += 32) dw = min(dw, sd[r]);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) dw = min(dw, __shfl_xor_sync(full, dw, off));
    int lw = rmin;
    for (;;) {
        const int i = lw - 1 - lane;
        const unsigned stop = __ballot_sync(full, i < 0 || sd[i] < dw);
        if (stop) {
            lw -= __ffs(stop) - 1;
            break;
        }
        lw -= 32;
    }
    int rw = rmax;
    for (;;) {
        const int i = rw + lane;
        const unsigned stop = __ballot_sync(full, i >= k - 1 || sd[i] < dw);
        if (stop) {
            rw += __ffs(stop) - 1;
            break;
        }
        rw += 32;
    }
    // Hartigan over the leaves [lw, rw] of w, left to right: leaf r, then the gap after it closes the open nodes
    // deeper than it and joins or opens the node at its depth; the gap after rw closes them all
    int2 *stk = reinterpret_cast<int2 *>(smem) + static_cast<int64_t>(warp) * stride;
    int top = -1, cost = 0, cur = 0;
    for (int base = lw; base <= rw; base += 32) {
        const int r = base + lane;
        int dep = -1, one = 0;
        if (r <= rw) {
            const int qr = sq[r];
            one = qr >= lo && qr <= hi;
            if (r < rw) dep = sd[r];
        }
        const int n = min(32, rw - base + 1);
        for (int i = 0; i < n; ++i) {
            const int dg = __shfl_sync(full, dep, i), s1 = __shfl_sync(full, one, i);
            if (lane != 0) continue;
            cur = s1 ? -1 : 1;
            while (top >= 0 && stk[top].x > dg) {
                cost += mp_attach(stk[top].y, cur);
                cur = (stk[top].y > 0) - (stk[top].y < 0);
                --top;
            }
            if (dg < 0) break;  // past rw: cur is w's sign
            if (top < 0 || stk[top].x < dg) stk[++top] = make_int2(dg, 0);
            cost += mp_attach(stk[top].y, cur);
        }
    }
    if (lane == 0) len[q] = cost + (cur < 0);
}

// One warp per tree of the chunk: k, and over its gaps the characters, their summed length and those of length 1.
__global__ void mp_reduce(TripletArgs a) {
    const int64_t w = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= a.t1 - a.t0) return;
    const int k = a.k[w];
    const int32_t *len = a.len + (a.leaf_off[a.t0 + w] - a.leaf0);
    long long s[3] = {0, 0, 0};
    if (k >= 3)
        for (int q = lane; q < k - 1; q += 32) {
            const int l = len[q];
            s[0] += l > 0;
            s[1] += l;
            s[2] += l == 1;
        }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1)
        for (int c = 0; c < 3; ++c) s[c] += __shfl_down_sync(0xffffffffu, s[c], off);
    if (lane == 0) {
        int64_t *o = a.per_tree + 4 * static_cast<int64_t>(a.t0 + w);
        o[0] = k;
        o[1] = s[0];
        o[2] = s[1];
        o[3] = s[2];
    }
}

// What both entry points share: the supertree validated and in pre-order, the depth of its leaves and the sparse
// table over the depths between consecutive leaves, the chunk plan, and on the device the source forest, its tours,
// those supertree arrays and the per-leaf scratch of a chunk.
struct TripletPass {
    PreorderTree s;
    int taxa = 0, T = 0, stride = 0, warps = 0;
    size_t row_smem = 0;
    std::vector<int32_t> leaf_depth, stab;
    std::vector<int> chunk_begin{0};
    int64_t most_leaves = 0, most_trees = 0;
    DevForest forest;
    DevTours tours;
    GrowBuf ident, flags, pos, d_leaf_depth, d_stab, qpos, spos, td, kbuf, rows;

    // Host side; returns the failure status (message set) or SCS_OK.  arrays: ints of (max depth + 1) per row warp
    // in shared memory, which `what` names in the message for a supertree too deep for them; tree_bytes: device bytes
    // per tree of a chunk on top of the per-leaf scratch.
    int prepare(scs_ctx *ctx, const char *name, const scs_forest *sources, int64_t num_nodes, const int32_t *parent,
                const int32_t *taxon, int arrays, size_t tree_bytes,
                const char *what = "the shared-memory Fenwick tree of a row") {
        taxa = sources->num_taxa;
        if (preorder_supertree(num_nodes, parent, taxon, taxa, &s))
            return fail(ctx, SCS_ERR_INPUT, (std::string(name) + ": malformed supertree (parent[i] >= i, a tip without a "
                                             "taxon of the forest, or a repeated taxon)").c_str());
        const int n = static_cast<int>(num_nodes), NL = s.leaves;
        T = sources->num_trees();
        // depth of every leaf and of the LCA of consecutive leaves: in pre-order the node after a tip hangs off that LCA
        std::vector<int32_t> depth(static_cast<size_t>(n), 0), adj(static_cast<size_t>(std::max(NL - 1, 1)), 0);
        leaf_depth.assign(static_cast<size_t>(NL), 0);
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
        stab.assign(static_cast<size_t>(levels) * NL, 0);
        std::copy(adj.begin(), adj.begin() + std::max(NL - 1, 0), stab.begin());
        for (int l = 1; l < levels; ++l)
            for (int i = 0; i + (1 << l) <= NL - 1; ++i)
                stab[static_cast<size_t>(l) * NL + i] = std::min(stab[static_cast<size_t>(l - 1) * NL + i],
                                                                 stab[static_cast<size_t>(l - 1) * NL + i + (1 << (l - 1))]);
        // per row warp: `arrays` arrays of max_depth + 1 ints in shared memory (Fenwick trees, histograms)
        stride = max_depth + 1;
        const size_t warp_smem = static_cast<size_t>(arrays) * stride * sizeof(int32_t);
        warps = static_cast<int>(std::min<size_t>(kMaxRowWarps, ctx->smem_optin / warp_smem));
        if (warps < 1)
            return fail(ctx, SCS_ERR_INVALID, (std::string(name) + ": the supertree is too deep for " + what).c_str());
        row_smem = static_cast<size_t>(warps) * warp_smem;

        const std::vector<int64_t> &loff = sources->leaf_offsets;
        for (int t = 0; t < T;) {
            const int b = chunk_begin.back();
            int e = t + 1;
            while (e < T && static_cast<size_t>(loff[e + 1] - loff[b]) * kLeafScratch <= kScratchBytes &&
                   static_cast<size_t>(e + 1 - b) * tree_bytes <= kMatrixBytes)
                ++e;
            most_leaves = std::max(most_leaves, loff[e] - loff[b]);
            most_trees = std::max<int64_t>(most_trees, e - b);
            chunk_begin.push_back(e);
            t = e;
        }
        return SCS_OK;
    }

    // Uploads and scratch; fills the fields of `args` that do not change from chunk to chunk.
    int upload(scs_ctx *ctx, const scs_forest *sources, TripletArgs *args) {
        int rc;
        if ((rc = devforest_upload(ctx, sources, 0, &forest))) return rc;
        std::vector<int32_t> identity(static_cast<size_t>(taxa > 0 ? taxa : 1));
        for (size_t x = 0; x < identity.size(); ++x) identity[x] = static_cast<int32_t>(x);
        if ((rc = put(ctx, ident, identity.data(), identity.size() * sizeof(int32_t))) ||
            (rc = put(ctx, pos, s.pos.data(), s.pos.size() * sizeof(int32_t))) ||
            (rc = put(ctx, d_leaf_depth, leaf_depth.data(), leaf_depth.size() * sizeof(int32_t))) ||
            (rc = put(ctx, d_stab, stab.data(), stab.size() * sizeof(int32_t))))
            return rc;
        if ((rc = grow(ctx, flags, 2 * sizeof(int32_t)))) return rc;
        SCS_CUDA(ctx, cudaMemsetAsync(flags.ptr, 0, 2 * sizeof(int32_t), ctx->stream));
        if ((rc = devforest_tours(ctx, forest, 0, ident.as<int32_t>(), &tours, flags.as<int32_t>()))) return rc;
        const size_t L = static_cast<size_t>(most_leaves) + 1;
        if ((rc = grow(ctx, qpos, L * 4)) || (rc = grow(ctx, spos, L * 4)) || (rc = grow(ctx, td, L * 4)) ||
            (rc = grow(ctx, rows, L * 4 * sizeof(int64_t))) || (rc = grow(ctx, kbuf, static_cast<size_t>(most_trees) * 4)))
            return rc;
        args->taxa = taxa;
        args->n_leaves = s.leaves;
        args->pos = pos.as<int32_t>();
        args->leaf_depth = d_leaf_depth.as<int32_t>();
        args->stab = d_stab.as<int32_t>();
        args->leaf_off = forest.leaf_off.as<int64_t>();
        args->leaf_taxon = tours.leaf_taxon.as<int32_t>();
        args->adj_depth = tours.adj_depth.as<int32_t>();
        args->qpos = qpos.as<int32_t>();
        args->spos = spos.as<int32_t>();
        args->td = td.as<int32_t>();
        args->k = kbuf.as<int32_t>();
        args->rows = rows.as<int64_t>();
        return SCS_OK;
    }

    // Points `args` at chunk c and runs tp_prep on it.
    int prep_chunk(scs_ctx *ctx, const scs_forest *sources, size_t c, TripletArgs *args) {
        const std::vector<int64_t> &loff = sources->leaf_offsets;
        const int b = chunk_begin[c], e = chunk_begin[c + 1];
        args->t0 = b;
        args->t1 = e;
        args->leaf0 = loff[b];
        args->chunk_leaves = loff[e] - loff[b];
        tp_prep<<<e - b, kPrepThreads, 0, ctx->stream>>>(*args);
        SCS_LAUNCHED(ctx, "tp_prep");
        return SCS_OK;
    }

    static int put(scs_ctx *ctx, GrowBuf &buf, const void *src, size_t bytes) {
        int r;
        if ((r = grow(ctx, buf, bytes))) return r;
        SCS_CUDA(ctx, cudaMemcpyAsync(buf.ptr, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
        return SCS_OK;
    }

    void release_all(scs_ctx *ctx) {
        forest.free_all(ctx);
        tours.free_all(ctx);
        for (GrowBuf *b : {&ident, &flags, &pos, &d_leaf_depth, &d_stab, &qpos, &spos, &td, &kbuf, &rows}) release(ctx, *b);
    }
};

}  // namespace
}  // namespace scs

using namespace scs;

extern "C" int scs_supertree_triplets(scs_ctx *ctx, const scs_forest *sources, int64_t num_nodes, const int32_t *parent,
                                      const int32_t *taxon, int64_t *per_tree) {
    if (!ctx) return SCS_ERR_INVALID;
    if (!sources || !parent || !taxon || !per_tree || num_nodes <= 0 || num_nodes >= (int64_t(1) << 31))
        return fail(ctx, SCS_ERR_INVALID, "scs_supertree_triplets: bad argument");
    TripletPass p;
    int rc = p.prepare(ctx, "scs_supertree_triplets", sources, num_nodes, parent, taxon, 2, 0);
    if (rc) return rc;
    const int T = p.T, taxa = p.taxa;
    std::fill(per_tree, per_tree + 5 * static_cast<int64_t>(T), 0);
    if (T == 0) return SCS_OK;

    GrowBuf d_per_tree;
    auto run = [&]() -> int {
        TripletArgs args{};
        if ((rc = p.upload(ctx, sources, &args))) return rc;
        if ((rc = grow(ctx, d_per_tree, 5 * static_cast<size_t>(T) * sizeof(int64_t)))) return rc;
        if (p.row_smem > 48 * 1024)
            SCS_CUDA(ctx, cudaFuncSetAttribute(tp_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(p.row_smem)));
        args.per_tree = d_per_tree.as<int64_t>();
        for (size_t c = 0; c + 1 < p.chunk_begin.size(); ++c) {
            if ((rc = p.prep_chunk(ctx, sources, c, &args))) return rc;
            if (args.chunk_leaves > 0) {
                tp_rows<<<ceil_div(args.chunk_leaves, p.warps), p.warps * 32, p.row_smem, ctx->stream>>>(args, p.stride);
                SCS_LAUNCHED(ctx, "tp_rows");
            }
            tp_reduce<<<ceil_div(args.t1 - args.t0, 8), 256, 0, ctx->stream>>>(args);
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
                per_tree[5 * static_cast<int64_t>(t)] = x >= 0 && x < taxa && p.s.pos[x] >= 0;
            }
        return SCS_OK;
    };
    rc = run();
    p.release_all(ctx);
    release(ctx, d_per_tree);
    cudaStreamSynchronize(ctx->stream);
    return rc;
}

extern "C" int scs_supertree_taxon_triplets(scs_ctx *ctx, const scs_forest *sources, int64_t num_nodes,
                                            const int32_t *parent, const int32_t *taxon, int64_t *per_taxon,
                                            double *weighted) {
    if (!ctx) return SCS_ERR_INVALID;
    if (!sources || !parent || !taxon || !per_taxon || num_nodes <= 0 || num_nodes >= (int64_t(1) << 31))
        return fail(ctx, SCS_ERR_INVALID, "scs_supertree_taxon_triplets: bad argument");
    const int64_t taxa = sources->num_taxa;
    TripletPass p;
    int rc = p.prepare(ctx, "scs_supertree_taxon_triplets", sources, num_nodes, parent, taxon, 3,
                       4 * static_cast<size_t>(taxa) * sizeof(int64_t));
    if (rc) return rc;
    const int T = p.T;
    std::fill(per_taxon, per_taxon + 6 * taxa, 0);
    if (weighted) std::fill(weighted, weighted + 3 * taxa, 0.0);
    if (T == 0 || taxa == 0) return SCS_OK;

    GrowBuf s_taxon, matrix, d_per_taxon, d_weighted;
    auto run = [&]() -> int {
        TripletArgs args{};
        if ((rc = p.upload(ctx, sources, &args))) return rc;
        std::vector<int32_t> taxon_at(static_cast<size_t>(std::max(p.s.leaves, 1)), 0);
        for (int64_t x = 0; x < taxa; ++x)
            if (p.s.pos[x] >= 0) taxon_at[p.s.pos[x]] = static_cast<int32_t>(x);
        const size_t matrix_bytes = static_cast<size_t>(p.most_trees) * 4 * taxa * sizeof(int64_t);
        if ((rc = TripletPass::put(ctx, s_taxon, taxon_at.data(), taxon_at.size() * sizeof(int32_t))) ||
            (rc = grow(ctx, matrix, matrix_bytes)) || (rc = grow(ctx, d_per_taxon, 6 * taxa * sizeof(int64_t))) ||
            (rc = grow(ctx, d_weighted, 3 * taxa * sizeof(double))))
            return rc;
        SCS_CUDA(ctx, cudaMemsetAsync(d_per_taxon.ptr, 0, 6 * taxa * sizeof(int64_t), ctx->stream));
        SCS_CUDA(ctx, cudaMemsetAsync(d_weighted.ptr, 0, 3 * taxa * sizeof(double), ctx->stream));
        if (p.row_smem > 48 * 1024)
            SCS_CUDA(ctx, cudaFuncSetAttribute(tx_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(p.row_smem)));
        args.s_taxon = s_taxon.as<int32_t>();
        args.weight = p.forest.weight.as<double>();
        args.matrix = matrix.as<int64_t>();
        args.per_taxon = d_per_taxon.as<int64_t>();
        args.weighted = d_weighted.as<double>();
        for (size_t c = 0; c + 1 < p.chunk_begin.size(); ++c) {
            if ((rc = p.prep_chunk(ctx, sources, c, &args))) return rc;
            const int trees = args.t1 - args.t0;
            SCS_CUDA(ctx, cudaMemsetAsync(matrix.ptr, 0xff, static_cast<size_t>(trees) * 4 * taxa * sizeof(int64_t), ctx->stream));
            if (args.chunk_leaves > 0) {
                SCS_CUDA(ctx, cudaMemsetAsync(p.rows.ptr, 0, 4 * static_cast<size_t>(args.chunk_leaves) * sizeof(int64_t), ctx->stream));
                tx_rows<<<ceil_div(args.chunk_leaves, p.warps), p.warps * 32, p.row_smem, ctx->stream>>>(args, p.stride);
                SCS_LAUNCHED(ctx, "tx_rows");
                tx_tree<<<ceil_div(trees, 8), 256, 0, ctx->stream>>>(args);
                SCS_LAUNCHED(ctx, "tx_tree");
            }
            tx_reduce<<<ceil_div(taxa, 256), 256, 0, ctx->stream>>>(args);
            SCS_LAUNCHED(ctx, "tx_reduce");
        }
        SCS_CUDA(ctx, cudaMemcpyAsync(per_taxon, d_per_taxon.ptr, 6 * taxa * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
        if (weighted)
            SCS_CUDA(ctx, cudaMemcpyAsync(weighted, d_weighted.ptr, 3 * taxa * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        ctx->d2h_bytes += static_cast<int64_t>(6 * taxa * sizeof(int64_t) + (weighted ? 3 * taxa * sizeof(double) : 0));
        return SCS_OK;
    };
    rc = run();
    p.release_all(ctx);
    for (GrowBuf *b : {&s_taxon, &matrix, &d_per_taxon, &d_weighted}) release(ctx, *b);
    cudaStreamSynchronize(ctx->stream);
    return rc;
}

extern "C" int scs_supertree_mrp(scs_ctx *ctx, const scs_forest *sources, int64_t num_nodes, const int32_t *parent,
                                 const int32_t *taxon, int64_t *per_tree) {
    if (!ctx) return SCS_ERR_INVALID;
    if (!sources || !parent || !taxon || !per_tree || num_nodes <= 0 || num_nodes >= (int64_t(1) << 31))
        return fail(ctx, SCS_ERR_INVALID, "scs_supertree_mrp: bad argument");
    TripletPass p;
    int rc = p.prepare(ctx, "scs_supertree_mrp", sources, num_nodes, parent, taxon, 2, 0,
                       "the shared-memory stack of a character");
    if (rc) return rc;
    const int T = p.T, taxa = p.taxa;
    const int words = (p.s.leaves + 31) / 32;
    const size_t rank_smem = static_cast<size_t>(words) * 8;
    if (rank_smem + 1024 > ctx->smem_optin)  // room for the static shared arrays
        return fail(ctx, SCS_ERR_INVALID, "scs_supertree_mrp: the supertree has too many tips for the shared-memory bitmap");
    std::fill(per_tree, per_tree + 4 * static_cast<int64_t>(T), 0);
    if (T == 0) return SCS_OK;

    GrowBuf d_per_tree;
    auto run = [&]() -> int {
        TripletArgs args{};
        if ((rc = p.upload(ctx, sources, &args))) return rc;
        if ((rc = grow(ctx, d_per_tree, 4 * static_cast<size_t>(T) * sizeof(int64_t)))) return rc;
        if (p.row_smem > 48 * 1024)
            SCS_CUDA(ctx, cudaFuncSetAttribute(mp_chars, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(p.row_smem)));
        if (rank_smem > 48 * 1024)
            SCS_CUDA(ctx, cudaFuncSetAttribute(mp_rank, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(rank_smem)));
        // four ints per tour position in the scratch of the triplet rows
        const int64_t L = p.most_leaves + 1;
        int32_t *scratch = p.rows.as<int32_t>();
        args.words = words;
        args.sq = scratch;
        args.sr = scratch + L;
        args.sdep = scratch + 2 * L;
        args.len = scratch + 3 * L;
        args.per_tree = d_per_tree.as<int64_t>();
        for (size_t c = 0; c + 1 < p.chunk_begin.size(); ++c) {
            if ((rc = p.prep_chunk(ctx, sources, c, &args))) return rc;
            if (args.chunk_leaves > 0) {
                mp_rank<<<args.t1 - args.t0, kPrepThreads, rank_smem, ctx->stream>>>(args);
                SCS_LAUNCHED(ctx, "mp_rank");
                mp_chars<<<ceil_div(args.chunk_leaves, p.warps), p.warps * 32, p.row_smem, ctx->stream>>>(args, p.stride);
                SCS_LAUNCHED(ctx, "mp_chars");
            }
            mp_reduce<<<ceil_div(args.t1 - args.t0, 8), 256, 0, ctx->stream>>>(args);
            SCS_LAUNCHED(ctx, "mp_reduce");
        }
        const size_t out_bytes = 4 * static_cast<size_t>(T) * sizeof(int64_t);
        SCS_CUDA(ctx, cudaMemcpyAsync(per_tree, d_per_tree.ptr, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        ctx->d2h_bytes += static_cast<int64_t>(out_bytes);
        // a lone tip has no tour: it shares one taxon with S or none
        const std::vector<int64_t> &noff = sources->node_offsets;
        for (int t = 0; t < T; ++t)
            if (noff[t + 1] - noff[t] == 1) {
                const int x = sources->taxon[noff[t]];
                per_tree[4 * static_cast<int64_t>(t)] = x >= 0 && x < taxa && p.s.pos[x] >= 0;
            }
        return SCS_OK;
    };
    rc = run();
    p.release_all(ctx);
    release(ctx, d_per_tree);
    cudaStreamSynchronize(ctx->stream);
    return rc;
}
