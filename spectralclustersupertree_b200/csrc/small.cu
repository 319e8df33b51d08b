// One-CTA path for small recursion nodes (n <= 64 vertices).
//
// Three quarters of the recursion nodes of a supertree job have fewer than 32 taxa; on them the
// staged path (components, contraction, Lanczos, 2-means: dozens of launches and several host
// round trips) is pure latency.  Here everything after the graph build -- the reference's
// _get_graph_components (/root/reference/src/sc_supertree/scs.py:458-492),
// _contract_proper_cluster_graph (:261-387) and spectral_cluster_graph (:210-258) -- runs in one
// launch of one CTA with the graph in shared memory, and the host reads one small record back.
//
//  * components: transitive closure of the 64-bit adjacency rows by repeated squaring;
//  * contraction: the same closure on the max-graph rows, then a max-merge of the weights;
//  * spectral: N = D^-1/2 W D^-1/2 is formed explicitly and diagonalised by a parallel cyclic
//    Jacobi iteration (round-robin pair ordering).  The known eigenpair (1, sqrt(d)) is moved out
//    of the way with M = N - 2 q0 q0^T, so the Fiedler pair is the largest eigenpair of M and the
//    next eigenvalue is exact as well (exact repeated-eigenvalue detection);
//  * sign flip and exact 1-D 2-means as in spectral.cu.

#include <algorithm>
#include <numeric>

#include "common.cuh"

namespace scs {

namespace {

constexpr int kThreads = 256;  // fixed for both capacities: the Jacobi convergence sums are associated by it
constexpr int kWarps = kThreads / 32;
constexpr double kGapTie = 1e-7;
constexpr double kMarginTie = 1e-9;

// A chunk of a node's source trees staged for the graph build: their tours in input order, concatenated.
template <int CAP>
struct TourChunk {
    static constexpr int kLeaves = 16 * CAP;  // a chunk always takes at least one well-formed tree (k <= n <= CAP)
    static constexpr int kTrees = kThreads;   // one thread per tree reads the offsets: at most kThreads trees
    static constexpr int kLevels = CAP == 32 ? 4 : 5;  // sparse-table levels 1 .. kLevels cover gap runs up to CAP - 1
    int taxon[kLeaves], depth[kLeaves];
    double val[kLeaves];
    int start[kTrees], k[kTrees], rd[kTrees];
    double w[kTrees];
    long long span[kLevels][kLeaves];  // span[L - 1][e]: the least gap key of gaps e .. e + 2^L - 1
};

template <int CAP>
struct SmallShared {
    double A[CAP][CAP + 1];  // W, then Wc, then M (padded: column sweeps hit distinct banks)
    union {
        struct {
            double V[CAP][CAP + 1];  // Jacobi eigenvectors
            double B[CAP][CAP + 1];  // the (contracted) weights the split was computed from: residual check
        };
        TourChunk<CAP> tours;        // graph build only (batched path), done before V and B are used
    };
    unsigned short cnt[CAP][CAP];    // co-occurrence counts (batched path: graph built in shared memory)
    int occ[CAP];
    double cs[CAP / 2][2];
    double deg[CAP], isd[CAP], q0[CAP], u[CAP], sorted[CAP];
    unsigned long long adj[CAP], mx[CAP], reach[CAP];
    int label[CAP], group[CAP], member_of[CAP], side[CAP];
    double red[2 * (kThreads / 32) + 2];
    int ired[4];
    long long clock_start;  // batched kernel, thread 0: profiling counters
};

// Two block sums at once, each associated as before: thread partials, a shuffle tree per warp, then the warp
// partials in order -- the Jacobi sweep count depends on these bits.
__device__ __forceinline__ void block_sum2_small(double &x, double &y, double *red) {
    constexpr int W = kThreads / 32;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        x += __shfl_down_sync(0xffffffffu, x, off);
        y += __shfl_down_sync(0xffffffffu, y, off);
    }
    __syncthreads();
    if ((threadIdx.x & 31) == 0) {
        red[threadIdx.x >> 5] = x;
        red[W + (threadIdx.x >> 5)] = y;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0, t = 0.0;
        for (int w = 0; w < W; ++w) s += red[w];
        for (int w = 0; w < W; ++w) t += red[W + w];
        red[2 * W] = s;
        red[2 * W + 1] = t;
    }
    __syncthreads();
    x = red[2 * W];
    y = red[2 * W + 1];
}

// reach[v] = bit set of the vertices connected to v (v included); label[v] = smallest of them
__device__ void closure(int n, const unsigned long long *rows, unsigned long long *reach, int *label) {
    const int v = threadIdx.x;
    if (v < n) reach[v] = rows[v] | (1ull << v);
    __syncthreads();
    for (int len = 1; len < n - 1; len <<= 1) {  // path lengths double every round, up to n - 1
        unsigned long long acc = 0;
        if (v < n) {
            unsigned long long bits = reach[v];
            acc = bits;
            while (bits) {
                const int b = __ffsll(static_cast<long long>(bits)) - 1;
                bits &= bits - 1;
                acc |= reach[b];
            }
        }
        __syncthreads();
        if (v < n) reach[v] = acc;
        __syncthreads();
    }
    if (v < n) label[v] = __ffsll(static_cast<long long>(reach[v])) - 1;
    __syncthreads();
}

// Pair k of round-robin round `step` over me (even) players, p < q; q == me - 1 >= m is a bye.
__device__ __forceinline__ void round_robin_pair(int me, int step, int k, int &p, int &q) {
    if (k == 0) { p = me - 1; q = step; }
    else { p = (step + k) % (me - 1); q = (step - k + (me - 1)) % (me - 1); }
    if (p > q) { const int t = p; p = q; q = t; }
}

// Everything after the graph build for one node whose weights are in S.A (n x n) and whose adjacency /
// max-graph rows are in S.adj / S.mx.  part, out, group_out, Wc_out are global pointers (the last two
// may be null).
template <int CAP>
__device__ void small_finish(SmallShared<CAP> &S, int n, int contract_edges, int32_t *__restrict__ part,
                             scs_node_stats *__restrict__ out, int32_t *__restrict__ group_out,
                             double *__restrict__ Wc_out) {
    const int tid = threadIdx.x;
    const double nan_v = __longlong_as_double(0x7ff8000000000000ll);

    // ---- components (scs.py:458-492) -----------------------------------------------------------
    closure(n, S.adj, S.reach, S.label);
    if (tid == 0) {
        int count = 0;
        for (int v = 0; v < n; ++v) {
            S.member_of[v] = count;  // rank of v among the representatives, valid where label[v] == v
            count += S.label[v] == v;
        }
        S.ired[0] = count;
    }
    __syncthreads();
    const int ncomp = S.ired[0];
    if (tid == 0) {
        out->n_components = ncomp;
        out->contracted_size = n;
        out->spectral_ran = 0;
        out->solver = 0;
        out->matvecs = 0;
        out->restarts = 0;
        out->tie_flag = 0;
        out->kmeans_stable_splits = 0;
        out->eig[0] = 0.0;
        out->eig[1] = nan_v;
        out->eig[2] = nan_v;
        out->residual = nan_v;
        out->margin = nan_v;
        out->kmeans_runner_up = 0.0;
    }
    if (ncomp != 1) {
        if (tid < n) part[tid] = S.member_of[S.label[tid]];
        return;
    }

    // ---- contraction (scs.py:261-387) ----------------------------------------------------------
    int m = n;
    if (contract_edges) {
        closure(n, S.mx, S.reach, S.label);
        if (tid == 0) {
            int count = 0;
            for (int v = 0; v < n; ++v) {
                S.member_of[v] = count;
                count += S.label[v] == v;
            }
            S.ired[1] = count;
        }
        __syncthreads();
        m = S.ired[1];
        if (tid < n) S.group[tid] = S.member_of[S.label[tid]];
        __syncthreads();
        if (m != n) {
            // Wc[A][B] = max over existing edges (u in A, v in B) of W[u][v]; staged in V as ordered keys
            for (int e = tid; e < m * m; e += kThreads) S.V[e / m][e % m] = __longlong_as_double(0ll);
            __syncthreads();
            for (int e = tid; e < n * n; e += kThreads) {
                const int u = e / n, v = e % n;
                if (!((S.adj[u] >> v) & 1ull)) continue;
                const int A = S.group[u], B = S.group[v];
                if (A == B) continue;  // edges inside a merged vertex vanish (scs.py:352-354)
                atomicMax(reinterpret_cast<unsigned long long *>(&S.V[A][B]), order_key(S.A[u][v]));
            }
            __syncthreads();
            for (int e = tid; e < m * m; e += kThreads) {
                const unsigned long long k = static_cast<unsigned long long>(__double_as_longlong(S.V[e / m][e % m]));
                S.V[e / m][e % m] = k ? order_value(k) : 0.0;
            }
            __syncthreads();
            for (int e = tid; e < m * m; e += kThreads) {
                S.A[e / m][e % m] = S.V[e / m][e % m];
                if (Wc_out) Wc_out[e] = S.V[e / m][e % m];
            }
            __syncthreads();
        }
        if (group_out && tid < n) group_out[tid] = S.group[tid];
    } else if (tid < n) {
        S.group[tid] = tid;
    }
    __syncthreads();
    if (tid == 0) {
        out->contracted_size = m;
        out->spectral_ran = 1;
    }
    if (m < 2) {
        if (tid == 0) out->solver = -1;  // nothing to split: the host raises SCS_ERR_TOO_SMALL
        return;
    }
    if (m == 2) {
        if (tid < n) part[tid] = S.group[tid];
        if (tid == 0) {
            out->solver = 1;
            out->eig[1] = 2.0;
            out->residual = 0.0;
            out->margin = 0.5;
        }
        return;
    }

    for (int e = tid; e < m * m; e += kThreads) S.B[e / m][e % m] = S.A[e / m][e % m];
    // ---- normalised affinity, trivial pair shifted away ------------------------------------------
    if (tid < m) {
        double d = 0.0;
        for (int j = 0; j < m; ++j) d += S.A[tid][j];
        S.deg[tid] = d;
    }
    __syncthreads();
    if (tid == 0) {
        double vol = 0.0;
        bool bad = false;
        for (int i = 0; i < m; ++i) {
            const double d = S.deg[i];
            if (!(d >= 0.0) || isinf(d)) bad = true;
            vol += d > 0.0 ? d : 0.0;
        }
        const double inv = vol > 0.0 ? 1.0 / sqrt(vol) : 0.0;
        for (int i = 0; i < m; ++i) {
            const double d = S.deg[i];
            const double s = d > 0.0 ? sqrt(d) : 0.0;
            S.isd[i] = d > 0.0 ? 1.0 / s : 1.0;
            S.q0[i] = s * inv;
        }
        S.ired[2] = bad;
    }
    __syncthreads();
    for (int e = tid; e < m * m; e += kThreads) {
        const int i = e / m, j = e % m;
        const double w = i == j ? 0.0 : S.A[i][j];  // scipy zeroes the diagonal (_laplacian.py:536-539)
        S.V[i][j] = S.isd[i] * w * S.isd[j] - 2.0 * S.q0[i] * S.q0[j];
    }
    __syncthreads();
    for (int e = tid; e < m * m; e += kThreads) {
        const int i = e / m, j = e % m;
        S.A[i][j] = 0.5 * (S.V[i][j] + S.V[j][i]);  // exactly symmetric
    }
    __syncthreads();
    for (int e = tid; e < m * m; e += kThreads) S.V[e / m][e % m] = (e / m == e % m) ? 1.0 : 0.0;
    __syncthreads();

    // ---- parallel cyclic Jacobi ------------------------------------------------------------------
    const int me = (m + 1) & ~1;  // even number of players; the extra one is a bye
    const int half = me >> 1;
    if (tid == 0) S.ired[1] = 0;  // sweeps done
    for (int sweep = 0; sweep < 30; ++sweep) {
        double off = 0.0, diag = 0.0;
        for (int e = tid; e < m * m; e += kThreads) {
            const int i = e / m, j = e % m;
            const double x = S.A[i][j];
            if (i == j) diag += x * x; else off += x * x;
        }
        block_sum2_small(off, diag, S.red);
        // off-diagonal Frobenius norm below 1e-14 of the whole: eigenvalues are then converged to
        // rounding (their error is quadratic in it) and eigenvectors to ~1e-14 / gap
        if (off <= 1e-28 * (diag + off) || off < 1e-300) break;
        if (tid == 0) S.ired[1] = sweep + 1;
        for (int step = 0; step < me - 1; ++step) {
            if (tid < half) {
                int p, q;
                round_robin_pair(me, step, tid, p, q);
                double c = 1.0, s = 0.0;
                if (q < m) {
                    const double apq = S.A[p][q];
                    if (fabs(apq) > 1e-300) {
                        const double tau = (S.A[q][q] - S.A[p][p]) / (2.0 * apq);
                        const double t = (tau >= 0.0 ? 1.0 : -1.0) / (fabs(tau) + sqrt(1.0 + tau * tau));
                        c = 1.0 / sqrt(1.0 + t * t);
                        s = t * c;
                    }
                }
                S.cs[tid][0] = c;
                S.cs[tid][1] = s;
            }
            __syncthreads();
            // columns: A <- A J, V <- V J
            for (int e = tid; e < m * half; e += kThreads) {
                const int r = e / half, k = e % half;
                int p, q;
                round_robin_pair(me, step, k, p, q);
                if (q >= m) continue;
                const double c = S.cs[k][0], s = S.cs[k][1];
                const double arp = S.A[r][p], arq = S.A[r][q];
                S.A[r][p] = c * arp - s * arq;
                S.A[r][q] = s * arp + c * arq;
                const double vrp = S.V[r][p], vrq = S.V[r][q];
                S.V[r][p] = c * vrp - s * vrq;
                S.V[r][q] = s * vrp + c * vrq;
            }
            __syncthreads();
            // rows: A <- J^T A
            for (int e = tid; e < m * half; e += kThreads) {
                const int r = e / half, k = e % half;
                int p, q;
                round_robin_pair(me, step, k, p, q);
                if (q >= m) continue;
                const double c = S.cs[k][0], s = S.cs[k][1];
                const double apr = S.A[p][r], aqr = S.A[q][r];
                S.A[p][r] = c * apr - s * aqr;
                S.A[q][r] = s * apr + c * aqr;
            }
            __syncthreads();
        }
    }

    // ---- Fiedler pair: largest eigenvalue of M (smallest index on exact ties) ------------------------
    if (tid == 0) {
        int best = 0;
        for (int i = 1; i < m; ++i)
            if (S.A[i][i] > S.A[best][best]) best = i;
        double second = -INFINITY;
        for (int i = 0; i < m; ++i)
            if (i != best && S.A[i][i] > second) second = S.A[i][i];
        S.ired[3] = best;
        S.red[0] = S.A[best][best];
        S.red[1] = second;
    }
    __syncthreads();
    const int col = S.ired[3];
    const double theta1 = S.red[0], theta2 = S.red[1];
    __syncthreads();

    // ---- embedding, sign flip, exact 1-D 2-means (see spectral.cu) ----------------------------------
    if (tid < m) S.u[tid] = S.V[tid][col] * S.isd[tid];
    __syncthreads();
    if (tid == 0) {
        int arg = 0;
        for (int i = 1; i < m; ++i)
            if (fabs(S.u[i]) > fabs(S.u[arg])) arg = i;
        const double sign = S.u[arg] < 0.0 ? -1.0 : 1.0;
        double mean = 0.0;
        for (int i = 0; i < m; ++i) {
            S.u[i] *= sign;
            mean += S.u[i];
        }
        S.red[2] = mean / m;
    }
    __syncthreads();
    if (tid < m) {  // rank sort (ties by index)
        const double x = S.u[tid];
        int rank = 0;
        for (int j = 0; j < m; ++j) rank += (S.u[j] < x) || (S.u[j] == x && j < tid);
        S.sorted[rank] = x;
    }
    __syncthreads();
    if (tid == 0) {
        const double mean = S.red[2];
        double all = 0.0;
        for (int i = 0; i < m; ++i) all += S.sorted[i] - mean;
        double prefix = 0.0, bscore = -1.0;
        int bi = 1;
        for (int i = 0; i + 1 < m; ++i) {
            prefix += S.sorted[i] - mean;
            const int cnt = i + 1;
            const double rest = all - prefix;
            const double score = prefix * prefix / cnt + rest * rest / (m - cnt);
            if (score > bscore) { bscore = score; bi = cnt; }
        }
        int stable = 0;
        double runner = -1.0, lower = 0.0;
        prefix = 0.0;
        for (int i = 0; i + 1 < m; ++i) {
            prefix += S.sorted[i] - mean;
            const int cnt = i + 1;
            if (cnt == bi) lower = prefix;
            const double rest = all - prefix;
            const double mid = mean + 0.5 * (prefix / cnt + rest / (m - cnt));
            if (S.sorted[i] < mid && mid < S.sorted[i + 1]) {
                stable += 1;
                if (cnt != bi) runner = fmax(runner, prefix * prefix / cnt + rest * rest / (m - cnt));
            }
        }
        const double c0 = mean + lower / bi;
        const double c1 = mean + (all - lower) / (m - bi);
        const double mid = 0.5 * (c0 + c1);
        const double range = fmax(S.sorted[m - 1] - S.sorted[0], 1e-300);
        const double margin = fmin(fabs(S.sorted[bi - 1] - mid), fabs(S.sorted[bi] - mid)) / range;
        S.red[3] = S.sorted[bi];
        out->solver = 2;
        out->matvecs = S.ired[1];  // Jacobi sweeps (the dense solver applies no matvec)
        out->eig[1] = 1.0 - theta1;
        out->eig[2] = 1.0 - theta2;
        out->margin = margin;
        out->kmeans_stable_splits = stable;
        out->kmeans_runner_up = (runner >= 0.0 && bscore > 0.0) ? runner / bscore : 0.0;
        int flag = 0;
        if (theta1 - theta2 < kGapTie) flag |= 1;
        if (!(margin >= kMarginTie)) flag |= 2;
        if (S.ired[2]) flag |= 8;
        if (stable > 1) flag |= 16;
        out->tie_flag = flag;
    }
    __syncthreads();
    const double threshold = S.red[3];
    if (tid < m) S.side[tid] = S.u[tid] >= threshold ? 1 : 0;
    __syncthreads();
    if (tid < n) part[tid] = S.side[S.group[tid]];

    // residual of the accepted pair against the operator it was computed from: |N y - theta y|
    if (tid < m) {
        double acc = 0.0;
        for (int j = 0; j < m; ++j)
            if (j != tid) acc += S.isd[tid] * S.B[tid][j] * S.isd[j] * S.V[j][col];
        acc -= theta1 * S.V[tid][col];
        S.deg[tid] = acc * acc;
    }
    __syncthreads();
    if (tid == 0) {
        double rr = 0.0;
        for (int i = 0; i < m; ++i) rr += S.deg[i];
        out->residual = sqrt(rr);
    }
}

// ---- per-node entry: graph already built in global memory (csrc/pcg.cu) ------------------------------
__global__ void __launch_bounds__(kThreads)
small_node_kernel(int n, int words, int contract_edges, const double *__restrict__ W,
                  const uint32_t *__restrict__ adj_bits, const uint32_t *__restrict__ max_bits,
                  int32_t *__restrict__ part, scs_node_stats *__restrict__ out,
                  int32_t *__restrict__ group_out, double *__restrict__ Wc_out) {
    extern __shared__ __align__(16) unsigned char raw[];
    SmallShared<kSmallNode> &S = *reinterpret_cast<SmallShared<kSmallNode> *>(raw);
    const int tid = threadIdx.x;
    for (int e = tid; e < n * n; e += kThreads) S.A[e / n][e % n] = W[e];
    if (tid < n) {
        unsigned long long a = adj_bits[static_cast<size_t>(tid) * words];
        unsigned long long m = max_bits ? max_bits[static_cast<size_t>(tid) * words] : 0ull;
        if (words > 1) {
            a |= static_cast<unsigned long long>(adj_bits[static_cast<size_t>(tid) * words + 1]) << 32;
            if (max_bits) m |= static_cast<unsigned long long>(max_bits[static_cast<size_t>(tid) * words + 1]) << 32;
        }
        S.adj[tid] = a;
        S.mx[tid] = m;
    }
    __syncthreads();
    small_finish(S, n, contract_edges, part, out, group_out, Wc_out);
}

// Cycle counters of the batched kernel, summed over its CTAs: [0] graph build, [1] everything after it (profiling aid:
// scs_debug_small_cycles).
__device__ unsigned long long g_small_cycles[2];

// (depth, position) of the gap after chunk position e, ordered so that the minimum is the leftmost shallowest gap
__device__ __forceinline__ long long gap_key(int depth, int e) {
    return static_cast<long long>(depth) * 4294967296ll + e;
}

// least gap key over gaps e .. e + 2^L - 1 of the staged chunk
template <int CAP>
__device__ __forceinline__ long long span_key(const TourChunk<CAP> &C, int L, int e) {
    return L == 0 ? gap_key(C.depth[e], e) : C.span[L - 1][e];
}

// ---- batched entry: one CTA per node builds the node's graph from its leaf tours in shared memory
//      (the reference's _proper_cluster_graph_edges, scs.py:495-663) and finishes it ------------------
// The node's trees are staged in chunks, and a sparse table of the gap keys (least key over every run of 2^L gaps) is
// built over each chunk: a few barriers per chunk, none per tree.  Warp w owns the rows a with a % kWarps == w (their
// W and count cells and occ[a]) and walks the chunk's trees in input order; for a row at tour position p of a tree,
// lane l holds positions l*E .. l*E + E - 1, and two table entries give every other position j the leftmost
// shallowest gap between p and j: the LCA of the two leaves.  Entries that run past a tree's last gap are never read
// (a query stays inside the gaps between the two leaves).  So every W entry
// receives its terms in tree order with separately rounded multiply and add -- the same sums, bit for bit, as
// pcg_rows_kernel and the reference -- and both triangles are built directly.
// order (may be null: identity) lists the batch's nodes in launch order; CTA b runs node order[first + b].
template <int CAP>
__global__ void __launch_bounds__(kThreads, CAP == 32 ? 4 : 2)
small_batch_kernel(const scs_small_node *__restrict__ nodes, const int32_t *__restrict__ order, int first,
                   const int64_t *__restrict__ leaf_offsets, const int32_t *__restrict__ leaf_taxon,
                   const int32_t *__restrict__ adj_depth, const double *__restrict__ adj_val,
                   const int32_t *__restrict__ root_depth, const double *__restrict__ tree_weight, int contract_edges,
                   int32_t *__restrict__ part, scs_node_stats *__restrict__ stats, int32_t *__restrict__ bad,
                   int absolute_offsets) {
    constexpr int E = CAP / 32;  // tour positions per lane
    constexpr int kLeaves = TourChunk<CAP>::kLeaves;
    extern __shared__ __align__(16) unsigned char raw[];
    SmallShared<CAP> &S = *reinterpret_cast<SmallShared<CAP> *>(raw);
    TourChunk<CAP> &C = S.tours;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = order ? order[first + blockIdx.x] : first + static_cast<int>(blockIdx.x);
    const scs_small_node node = nodes[b];
    const int n = node.n;
    if (tid == 0) S.clock_start = clock64();
    if (node.num_trees > kSmallMaxTrees || n < 1 || n > CAP) {
        // the co-occurrence counts are 16-bit here (the staged path switches to 32-bit counts at 65 536 trees,
        // pcg.cu `narrow`); the host entry points route such nodes to the staged path -- refuse loudly if one
        // arrives anyway
        if (tid == 0) {
            *bad = 1;
            stats[b].solver = -1;
        }
        return;
    }
    for (int e = tid; e < n * n; e += kThreads) {
        S.A[e / n][e % n] = 0.0;
        S.cnt[e / n][e % n] = 0;
    }
    if (tid < n) S.occ[tid] = 0;
    // T + 1 offsets per node, relative to its first leaf -- or the forest's absolute offsets
    const int64_t *offs = leaf_offsets + node.tree_base + (absolute_offsets ? 0 : b);
    const int64_t leaf_base = absolute_offsets ? 0 : node.leaf_base;
    for (int t0 = 0; t0 < node.num_trees;) {
        // the chunk: trees t0 .. t0 + count - 1, as many as have their leaves within kLeaves of the chunk's first
        const int64_t begin = offs[t0];
        const int t = t0 + tid;
        const bool fits = t < node.num_trees && offs[t + 1] - begin <= kLeaves;
        const int count = __syncthreads_count(fits);  // also: the previous chunk is done with the staging area
        if (count == 0) {  // one tree longer than a chunk has more leaves than vertices: malformed input
            if (tid == 0) *bad = 1;
            ++t0;
            continue;
        }
        if (tid < count) {
            C.start[tid] = static_cast<int>(offs[t] - begin);
            C.k[tid] = static_cast<int>(offs[t + 1] - offs[t]);
            C.w[tid] = tree_weight[node.tree_base + t];
            C.rd[tid] = root_depth[node.tree_base + t];
        }
        const int total = static_cast<int>(offs[t0 + count] - begin);
        for (int e = tid; e < total; e += kThreads) {
            const int64_t g = leaf_base + begin + e;
            const int a = leaf_taxon[g];
            C.taxon[e] = a;
            C.depth[e] = adj_depth[g];
            C.val[e] = adj_val[g];
            if (a < 0 || a >= n) *bad = 1;
        }
        __syncthreads();
        for (int L = 1; L <= TourChunk<CAP>::kLevels; ++L) {
            const int h = 1 << (L - 1);
            for (int e = tid; e < total; e += kThreads)
                C.span[L - 1][e] = min(span_key(C, L - 1, e), span_key(C, L - 1, min(e + h, total - 1)));
            __syncthreads();
        }
        for (int i = 0; i < count; ++i) {  // trees in input order
            const int k = C.k[i];
            if (k > n) {  // more leaves than vertices: malformed input
                if (tid == 0) *bad = 1;
                continue;
            }
            const int base = C.start[i], rd = C.rd[i];
            const double w = C.w[i];
            int tx[E];
            unsigned rows[E];
#pragma unroll
            for (int e = 0; e < E; ++e) {
                const int j = lane * E + e;
                tx[e] = j < k ? C.taxon[base + j] : -1;
                rows[e] = __ballot_sync(0xffffffffu, tx[e] >= 0 && tx[e] < n && tx[e] % kWarps == warp);
            }
#pragma unroll
            for (int e0 = 0; e0 < E; ++e0) {
                for (unsigned bits = rows[e0]; bits; bits &= bits - 1) {
                    const int p = (__ffs(bits) - 1) * E + e0;  // the row's tour position
                    const int a = C.taxon[base + p];
                    if (lane == 0) S.occ[a] += 1;
#pragma unroll
                    for (int e = 0; e < E; ++e) {
                        const int j = lane * E + e;
                        const int bj = tx[e];
                        if (j == p || bj < 0 || bj >= n) continue;
                        // gaps lo .. hi - 1 lie between the two leaves: two overlapping runs of 2^L gaps cover them
                        const int lo = base + min(j, p), hi = base + max(j, p);
                        const int L = 31 - __clz(hi - lo);
                        const long long kk = min(span_key(C, L, lo), span_key(C, L, hi - (1 << L)));
                        const int depth = static_cast<int>(kk >> 32);
                        if (depth == rd) continue;  // the LCA is the root: no edge (scs.py:552-556)
                        const int at = static_cast<int>(kk & 0xffffffffll);
                        S.A[a][bj] = __dadd_rn(S.A[a][bj], __dmul_rn(C.val[at], w));
                        S.cnt[a][bj] += 1;
                    }
                }
            }
        }
        t0 += count;
    }
    __syncthreads();
    if (tid < n) {
        unsigned long long a = 0, m = 0;
        const int occ_a = S.occ[tid];
        for (int c = 0; c < n; ++c) {
            const int k = S.cnt[tid][c];
            if (k > 0) {
                a |= 1ull << c;
                if (k == max(occ_a, S.occ[c])) m |= 1ull << c;
            }
        }
        S.adj[tid] = a;
        S.mx[tid] = contract_edges ? m : 0ull;
    }
    __syncthreads();
    if (tid == 0) {
        const long long clock_built = clock64();
        atomicAdd(&g_small_cycles[0], static_cast<unsigned long long>(clock_built - S.clock_start));
        S.clock_start = clock_built;
    }
    small_finish(S, n, contract_edges, part + node.vertex_base, stats + b, nullptr, nullptr);
    if (tid == 0) atomicAdd(&g_small_cycles[1], static_cast<unsigned long long>(clock64() - S.clock_start));
}

template <int CAP>
int launch_small_batch(scs_ctx *ctx, int count, int first, const scs_small_node *nodes_dev, const int32_t *order_dev,
                       const int64_t *leaf_offsets, const int32_t *leaf_taxon, const int32_t *adj_depth,
                       const double *adj_val, const int32_t *root_depth, const double *tree_weight, int contract_edges,
                       int32_t *part_dev, scs_node_stats *stats_dev, int32_t *bad_dev, int absolute_offsets) {
    if (count <= 0) return SCS_OK;
    small_batch_kernel<CAP><<<count, kThreads, sizeof(SmallShared<CAP>), ctx->stream>>>(
        nodes_dev, order_dev, first, leaf_offsets, leaf_taxon, adj_depth, adj_val, root_depth, tree_weight,
        contract_edges, part_dev, stats_dev, bad_dev, absolute_offsets);
    SCS_LAUNCHED(ctx, "small_batch_kernel");
    return SCS_OK;
}

}  // namespace

int small_node(scs_ctx *ctx, int n, int contract_edges, const double *W, const uint32_t *adj_bits,
               const uint32_t *max_bits, int32_t *part, scs_node_stats *out_dev, int32_t *group_out,
               double *Wc_out) {
    if (n < 1 || n > kSmallNode) return fail(ctx, SCS_ERR_INVALID, "small_node: size out of range");
    const size_t smem = sizeof(SmallShared<kSmallNode>);
    if (!ctx->small_configured) {
        SCS_CUDA(ctx, cudaFuncSetAttribute(small_node_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           static_cast<int>(smem)));
        ctx->small_configured = true;
    }
    small_node_kernel<<<1, kThreads, smem, ctx->stream>>>(n, scs_bit_words(n), contract_edges, W, adj_bits,
                                                         contract_edges ? max_bits : nullptr, part, out_dev, group_out,
                                                         Wc_out);
    SCS_LAUNCHED(ctx, "small_node_kernel");
    return SCS_OK;
}

int small_cycles(scs_ctx *ctx, unsigned long long *out2, int reset) {
    SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    SCS_CUDA(ctx, cudaMemcpyFromSymbol(out2, g_small_cycles, 2 * sizeof(unsigned long long)));
    if (reset) {
        const unsigned long long zero[2] = {0, 0};
        SCS_CUDA(ctx, cudaMemcpyToSymbol(g_small_cycles, zero, sizeof(zero)));
    }
    return SCS_OK;
}

int small_order(int num_nodes, const scs_small_node *nodes, int32_t *order) {
    std::iota(order, order + num_nodes, 0);
    const auto cost = [nodes](int32_t b) { return static_cast<int64_t>(nodes[b].n) * nodes[b].n * nodes[b].num_trees; };
    std::stable_sort(order, order + num_nodes, [&](int32_t x, int32_t y) {
        const bool bx = nodes[x].n > kSmallCap32, by = nodes[y].n > kSmallCap32;
        return bx != by ? by : cost(x) > cost(y);
    });
    int count = 0;
    for (int b = 0; b < num_nodes; ++b) count += nodes[b].n <= kSmallCap32;
    return count;
}

int small_batch(scs_ctx *ctx, int num_nodes, const scs_small_node *nodes_dev, const int32_t *order_dev, int num_cap32,
                const int64_t *leaf_offsets, const int32_t *leaf_taxon, const int32_t *adj_depth, const double *adj_val,
                const int32_t *root_depth, const double *tree_weight, int contract_edges, int32_t *part_dev,
                scs_node_stats *stats_dev, int32_t *bad_dev, int absolute_offsets) {
    if (num_nodes <= 0) return SCS_OK;
    if (!order_dev) num_cap32 = 0;  // launch order unknown on the host: every node takes the 64-capacity kernel
    if (!ctx->batch_configured) {
        SCS_CUDA(ctx, cudaFuncSetAttribute(small_batch_kernel<kSmallCap32>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           static_cast<int>(sizeof(SmallShared<kSmallCap32>))));
        SCS_CUDA(ctx, cudaFuncSetAttribute(small_batch_kernel<kSmallNode>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           static_cast<int>(sizeof(SmallShared<kSmallNode>))));
        ctx->batch_configured = true;
    }
    int rc = launch_small_batch<kSmallCap32>(ctx, num_cap32, 0, nodes_dev, order_dev, leaf_offsets, leaf_taxon,
                                             adj_depth, adj_val, root_depth, tree_weight, contract_edges, part_dev,
                                             stats_dev, bad_dev, absolute_offsets);
    if (rc) return rc;
    return launch_small_batch<kSmallNode>(ctx, num_nodes - num_cap32, num_cap32, nodes_dev, order_dev, leaf_offsets,
                                          leaf_taxon, adj_depth, adj_val, root_depth, tree_weight, contract_edges,
                                          part_dev, stats_dev, bad_dev, absolute_offsets);
}

}  // namespace scs
