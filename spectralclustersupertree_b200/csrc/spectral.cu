// Spectral bipartition of the (contracted) proper cluster graph on the GPU.
//
// Replaces spectral_cluster_graph of the reference (/root/reference/src/sc_supertree/scs.py:210-258),
// i.e. sklearn.cluster.SpectralClustering(2, affinity="precomputed", assign_labels="kmeans"):
//   L = I - D^-1/2 W D^-1/2   (scipy csgraph.laplacian(normed=True): degree 0 is scaled by 1)
//   x_0, x_1 = eigenvectors of the two smallest eigenvalues (sklearn: shift-invert ARPACK after a
//              dense LU of L); embedding rows u_k = x_k / sqrt(d); sign flip; 2-means.
//
// Here nothing is factorised.  With N = D^-1/2 W D^-1/2 the smallest eigenpair of L is known in
// closed form (eigenvalue 0, x_0 = sqrt(d) / |sqrt(d)|), so the Fiedler pair is the LARGEST
// eigenpair of N on the orthogonal complement of x_0: Lanczos with full (twice-applied classical
// Gram-Schmidt) re-orthogonalisation against x_0 and the whole basis.  The operator is the fused
// matvec  y = isd .* (W (isd .* v))  -- W is read once per application, straight from HBM, in
// fp64 (the parity contract needs a 1e-3 tree-weight difference and 1e-6 eigenvalues to survive).
// The projected tridiagonal problem is solved on the device (Sturm multi-section + twisted
// factorisation), so the host only reads back a residual estimate to decide when to stop.
// u_0 is constant on a connected graph, so sklearn's 2-means on (u_0, u_1) is 1-D 2-means on the
// Fiedler coordinate; it is solved exactly (sort, prefix sums, best split) instead of by ten
// random Lloyd restarts, which makes the partition deterministic.

#include "common.cuh"
#include "shard.cuh"
#include "spectral_dev.cuh"

#include <cooperative_groups.h>

#include <algorithm>
#include <chrono>
#include <cmath>

namespace scs {

namespace {

using namespace specdev;
namespace cg = cooperative_groups;

// ---- degree and scaling ---------------------------------------------------------------------
// one warp per row: d[a] = sum_b W[a][b]   (scipy _laplacian.py:543: column sums of a symmetric matrix)
__global__ void row_sums(int m, const double *__restrict__ W, double *__restrict__ degree) {
    const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (row >= m) return;
    const double *w = W + static_cast<size_t>(row) * m;
    double acc = 0.0;
    for (int j = lane; j < m; j += 32) acc += w[j];
    acc = warp_sum(acc);
    if (lane == 0) degree[row] = acc;
}

// isd = 1/sqrt(d) (1 where d == 0, scipy _laplacian.py:544-545); q0 = sqrt(d)/|sqrt(d)|; one CTA.
// flags[0] is raised if a degree is negative or not finite (sklearn would produce NaNs there).
__global__ void __launch_bounds__(kOneCta)
prepare_scaling(int m, const double *__restrict__ degree, double *__restrict__ isd, double *__restrict__ q0,
                int32_t *__restrict__ flags) {
    specdev::prepare_scaling_body(m, degree, isd, q0, flags);
}

__global__ void scale_vector(int m, const double *__restrict__ isd, const double *__restrict__ x,
                             double *__restrict__ z) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < m) z[i] = isd[i] * x[i];
}

// A CTA of kMvThreads threads works on kMvThreads / kGroup rows, kGroup threads each:
//   kGroup = 32   a warp per row: short rows (m < 2048);
//   kGroup = 256  a CTA per row: long rows (tens of KB), many waves.
// 64 and 128 threads per row exist for tuning (SCS_MATVEC_GROUP); measured under ncu on the C4 nodes they are
// within noise of 256 at every size from 2362 to 8765 columns (tools/matvec_bench.py, profiles/README.md): a
// 45 MB matrix takes 13 us whatever the shape -- launch ramp and tail, not the row split, separate it from the
// 7 us of the HBM roofline.
// The partial sums of a row are combined in a fixed order (lanes by shuffle tree, then warps in order), the
// same in the single-GPU and in the row-sharded kernel, so both produce the same bits.
__host__ __device__ constexpr int mv_group_of(int m) { return m < 2048 ? 32 : kMvThreads; }

// Row `row` of W (stored at `Wrow`) times z, by the kGroup threads of the calling group; the result is valid
// in the group's first thread.  `part` holds kMvThreads / 32 doubles.
template <int kGroup>
__device__ __forceinline__ double group_row_dot(const double *__restrict__ Wrow, const double *__restrict__ z, int m,
                                                double *part) {
    const int t = threadIdx.x % kGroup, warp = threadIdx.x >> 5;
    double acc = row_dot_partial(Wrow, z, m, t, kGroup);
    acc = warp_sum(acc);
    if (kGroup == 32) return acc;
    if ((threadIdx.x & 31) == 0) part[warp] = acc;
    __syncthreads();
    double s = 0.0;
    if (t == 0) {
#pragma unroll
        for (int w = 0; w < kGroup / 32; ++w) s += part[warp + w];
    }
    return s;
}

template <int kGroup>
__global__ void __launch_bounds__(kMvThreads)
matvec_rows(int m, const double *__restrict__ W, const double *__restrict__ isd, const double *__restrict__ z,
            double *__restrict__ y, const int32_t *__restrict__ done) {
    __shared__ double part[kMvThreads / 32];
    if (done && *done) return;
    constexpr int kRows = kMvThreads / kGroup;
    const int row = blockIdx.x * kRows + threadIdx.x / kGroup;
    const bool live = row < m;
    // rows past the end redo the last row (every thread must reach the barrier in group_row_dot)
    const double s = group_row_dot<kGroup>(W + static_cast<size_t>(live ? row : m - 1) * m, z, m, part);
    if (live && threadIdx.x % kGroup == 0) y[row] = isd[row] * s;
}

int launch_matvec_single(scs_ctx *ctx, int m, const double *W, const double *isd, const double *z, double *y,
                         const int32_t *done);

// threads per row; SCS_MATVEC_GROUP (32 / 64 / 128 / 256) overrides the choice for rows of >= 2048 columns (tuning)
int matvec_group(int m) {
    static const int forced = [] {
        const char *env = std::getenv("SCS_MATVEC_GROUP");
        const int v = env ? std::atoi(env) : 0;
        return (v == 32 || v == 64 || v == 128 || v == 256) ? v : 0;
    }();
    return forced && m >= 2048 ? forced : mv_group_of(m);
}

// Row-sharded operator fused with its all-gather (one process per GPU, rows [row0, row0 + nrows) of
// W on this rank): every CTA computes entries of y into the `vec` buffer of this rank's exchange window; the
// last CTA to finish copies the slice into every peer's window over NVLink, raises this rank's flag in every
// window and then waits until every rank has raised its flag here, so when the kernel ends the whole
// vector is in this rank's window.  Every entry is computed by the same code whatever rank owns the row,
// so the assembled vector is bit-identical to the single-GPU matvec's.
// kWarpRows mirrors the single-GPU choice (one warp per row below 2048 columns, one CTA per row above), so
// that the summation order of every entry is the same in both paths.
template <int kGroup>
__global__ void __launch_bounds__(kMvThreads)
matvec_rows_allgather(int m, int row0, int nrows, const double *__restrict__ W, const double *__restrict__ isd,
                      const double *__restrict__ z, const PeerTable peers, size_t vec_offset,
                      unsigned long long epoch, unsigned long long timeout_ns, const int32_t *__restrict__ done) {
    __shared__ double part[kMvThreads / 32];
    __shared__ unsigned int last;
    if (done && *done) return;  // the same on every rank: nobody signals, nobody waits
    constexpr int kRows = kMvThreads / kGroup;
    const int local = blockIdx.x * kRows + threadIdx.x / kGroup;
    const bool live = local < nrows;
    const double s = group_row_dot<kGroup>(W + static_cast<size_t>(live ? local : nrows - 1) * m, z, m, part);
    // The entry goes into this rank's OWN window with an ordinary store and a device-scope fence.  (Storing it
    // into every peer's window from here needed a system-scope fence per CTA -- thousands of NVLink round trips per
    // launch, which is why two GPUs were no faster than one: 70 us against 72.)
    double *mine_vec = reinterpret_cast<double *>(peers.window[peers.rank] + vec_offset);
    if (live && threadIdx.x % kGroup == 0) {
        mine_vec[row0 + local] = isd[row0 + local] * s;
        __threadfence();
    }
    __syncthreads();  // every store of this CTA is fenced before its ticket is drawn
    if (threadIdx.x == 0) {
        ShardHeader *mine = reinterpret_cast<ShardHeader *>(peers.window[peers.rank]);
        last = atomicInc(&mine->ticket, gridDim.x - 1) == gridDim.x - 1;
    }
    __syncthreads();
    if (!last) return;
    // The last CTA forwards the finished slice to every peer with coalesced stores, fences once, raises this rank's
    // flag in every window and waits until every rank has raised its flag here.
    __threadfence();
    for (int step = 1; step < peers.world; ++step) {
        const int p = (peers.rank + step) % peers.world;
        double *theirs = reinterpret_cast<double *>(peers.window[p] + vec_offset) + row0;
        for (int i = threadIdx.x; i < nrows; i += kMvThreads) theirs[i] = __ldcg(mine_vec + row0 + i);
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x < 32) peer_signal_and_wait(peers, epoch, timeout_ns);
}

int launch_matvec(scs_ctx *ctx, int m, const double *W, const double *isd, const double *z, double **y,
                  const int32_t *done = nullptr, RowBlock rows = RowBlock()) {
    if (rows.sharded()) {
        // the result lands in the window (double-buffered); *y is redirected there
        const ShardState &sh = ctx->shard;
        const ShardMatvecTicket ticket = shard_next_matvec(ctx);
        PeerTable peers;
        for (int r = 0; r < kMaxPeers; ++r) peers.window[r] = sh.peer[r];
        peers.rank = sh.rank;
        peers.world = sh.world;
        const int nrows = rows.row1 - rows.row0;
        *y = reinterpret_cast<double *>(sh.window + ticket.vec_offset);
        if (nrows <= 0) return fail(ctx, SCS_ERR_INVALID, "sharded matvec: a rank owns no rows");
        if (m >= kProfileMinSize)
            profile_begin(ctx, PROFILE_MATVEC, 8.0 * nrows * m + 8.0 * m + 8.0 * nrows * (1 + sh.world), 2.0 * nrows * m);
#define SCS_MV_AG(G)                                                                                          \
    matvec_rows_allgather<G><<<ceil_div(nrows, kMvThreads / G), kMvThreads, 0, ctx->stream>>>(                \
        m, rows.row0, nrows, W, isd, z, peers, ticket.vec_offset, ticket.epoch, ticket.timeout_ns, done)
        switch (matvec_group(m)) {
        case 32: SCS_MV_AG(32); break;
        case 64: SCS_MV_AG(64); break;
        case 128: SCS_MV_AG(128); break;
        default: SCS_MV_AG(256); break;
        }
#undef SCS_MV_AG
        if (m >= kProfileMinSize) profile_end(ctx);
        SCS_LAUNCHED(ctx, "matvec_rows_allgather");
        return SCS_OK;
    }
    return launch_matvec_single(ctx, m, W, isd, z, *y, done);
}

int launch_matvec_single(scs_ctx *ctx, int m, const double *W, const double *isd, const double *z, double *y,
                         const int32_t *done) {
    // algorithmic bytes: W once + read z, isd, write y
    if (m >= kProfileMinSize) profile_begin(ctx, PROFILE_MATVEC, 8.0 * m * m + 24.0 * m, 2.0 * m * m);
#define SCS_MV(G) matvec_rows<G><<<ceil_div(m, kMvThreads / G), kMvThreads, 0, ctx->stream>>>(m, W, isd, z, y, done)
    switch (matvec_group(m)) {
    case 32: SCS_MV(32); break;
    case 64: SCS_MV(64); break;
    case 128: SCS_MV(128); break;
    default: SCS_MV(256); break;
    }
#undef SCS_MV
    if (m >= kProfileMinSize) profile_end(ctx);
    SCS_LAUNCHED(ctx, "matvec_rows");
    return SCS_OK;
}

// ---- Lanczos vector kernels ------------------------------------------------------------------
// start vector: uniform(-1, 1) from a counter-based generator (sklearn: random_state.uniform(-1, 1, n),
// _arpack.py:31-33)
__global__ void random_start(int m, uint64_t seed, double *__restrict__ w) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const uint64_t r = splitmix64(seed * 0xD1342543DE82EF95ull + static_cast<uint64_t>(i) + 1ull);
    w[i] = 2.0 * (static_cast<double>(r >> 11) * (1.0 / 9007199254740992.0)) - 1.0;
}

// ---- Lanczos step tail of a large node (m > kFusedMax): one launch of a thread-block cluster ------------------
// Everything of a step except the operator application: both classical Gram-Schmidt passes against the nb leading
// basis vectors, the norm, the next basis vector v_{j+1} and z = isd .* v_{j+1}, alpha_j / beta_j and, at check
// steps, the projected eigenproblem.  Its verdict is latched in state[1] (state[2] = the step), so that the
// launches queued behind it fall through, as lanczos_tail does for m <= kFusedMax.  The basis (a few MB) stays in
// L2; kStepCluster CTAs share the work and meet at cluster barriers, which also make the global stores of one
// phase visible to the next.  No cooperative launch and no grid-wide sync: the cluster is co-scheduled.
// The summation order of every value is fixed by the decomposition below, whatever the cluster size:
//   h[k] = basis[k] . w     by one CTA of kVecThreads threads (thread stride, then block_sum);
//   w[i] -= h[k] basis[k]i  one thread per element, k ascending;
//   |w|^2                   kOneCta virtual threads (stride kOneCta, warp sums, then the 32 warp sums), computed
//                           by every CTA from the whole of w, so that all of them scale by the same bits;
//   projected problem       tridiag_solve by kVecThreads threads of CTA 0.
// state: [0] breakdown step, [1] done, [2] step at which done was raised.
constexpr int kStepCluster = 8;
constexpr int kDots = 4;  // basis vectors a CTA dots with w in one sweep

__global__ void __cluster_dims__(kStepCluster, 1, 1) __launch_bounds__(kVecThreads, 1)
lanczos_step(int m, int j, int nb, int hj, int check, const double *__restrict__ basis, double *w,
             const double *__restrict__ isd, double *h1, double *h2, double *alpha, double *beta, double *next,
             double *z, int32_t *state, double *coef, double *ritz) {
    extern __shared__ double step_smem[];
    double *hs = step_smem;                 // [kMaxBasis + 8] coefficients of the current pass
    double *tri = hs + (kMaxBasis + 8);     // 5 (j + 2) doubles for the projected problem
    __shared__ double scratch[33];
    __shared__ int counts[kVecThreads];
    __shared__ double pair[4];
    if (state[1]) return;  // converged earlier in this chunk (written by an earlier launch: the same in every CTA)
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = static_cast<int>(cluster.block_rank());
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int first = rank * kVecThreads + tid, stride = kStepCluster * kVecThreads;
    for (int pass = 0; pass < 2; ++pass) {
        double *h = pass ? h2 : h1;
        // this CTA's vectors k = rank + q kStepCluster, kDots at a time in one sweep over w (independent sums)
        for (int k0 = rank; k0 < nb; k0 += kDots * kStepCluster) {
            const double *b[kDots];
            double acc[kDots];
#pragma unroll
            for (int q = 0; q < kDots; ++q) {
                const int k = min(k0 + q * kStepCluster, nb - 1);  // past the end: a duplicate, never stored
                b[q] = basis + static_cast<size_t>(k) * m;
                acc[q] = 0.0;
            }
#pragma unroll 2
            for (int i = tid; i < m; i += kVecThreads) {
                const double wi = w[i];
#pragma unroll
                for (int q = 0; q < kDots; ++q) acc[q] = fma(b[q][i], wi, acc[q]);
            }
#pragma unroll
            for (int q = 0; q < kDots; ++q) {
                const double sum = block_sum(acc[q], scratch);
                if (tid == 0 && k0 + q * kStepCluster < nb) h[k0 + q * kStepCluster] = sum;
            }
        }
        cluster.sync();
        for (int k = tid; k < nb; k += kVecThreads) hs[k] = h[k];
        __syncthreads();
        for (int i = first; i < m; i += stride) {
            double acc = w[i];
#pragma unroll 8
            for (int k = 0; k < nb; ++k) acc = fma(-hs[k], basis[static_cast<size_t>(k) * m + i], acc);
            w[i] = acc;
        }
        cluster.sync();
    }
    // |w|^2 as one CTA of kOneCta threads sums it: virtual thread q * kVecThreads + tid, warp q * 8 + warp
    constexpr int kVirtual = kOneCta / kVecThreads;
    static_assert(kOneCta == 32 * 32 && kVirtual * kVecThreads == kOneCta, "32 virtual warps of 32 threads");
#pragma unroll
    for (int q = 0; q < kVirtual; ++q) {
        double ss = 0.0;
        for (int i = q * kVecThreads + tid; i < m; i += kOneCta) ss = fma(w[i], w[i], ss);
        ss = warp_sum(ss);
        if (lane == 0) scratch[q * (kVecThreads / 32) + warp] = ss;
    }
    __syncthreads();
    if (warp == 0) {
        const double t = warp_sum(scratch[lane]);
        if (lane == 0) scratch[32] = t;
    }
    __syncthreads();
    const double bnorm = sqrt(scratch[32]);
    if (rank == 0 && tid == 0) {
        beta[j] = bnorm;
        if (j > 0) {
            alpha[j] = h1[hj] + h2[hj];
            if (bnorm <= kBreakdown && state[0] == 0) state[0] = j;
        } else {
            state[0] = 0;
        }
    }
    const double inv = bnorm > 0.0 ? 1.0 / bnorm : 0.0;
    for (int i = first; i < m; i += stride) {
        const double v = w[i] * inv;
        next[i] = v;
        z[i] = isd[i] * v;
    }
    if (rank != 0 || !check || j == 0) return;
    __syncthreads();  // alpha / beta / state written by thread 0 are read below
    tridiag_solve(j, alpha, beta, state, coef, ritz, tri, counts, pair);
    if (tid == 0) {
        ritz[5] = static_cast<double>(j);
        if (ritz[3] <= kBreakdown || ritz[2] <= kResidualTol) {
            state[1] = 1;
            state[2] = j;
        }
    }
}
constexpr size_t kStepSmem = (kMaxBasis + 8 + 5 * (kMaxBasis + 2)) * sizeof(double);

// ---- fused Lanczos step tail (m <= kFusedMax) -----------------------------------------------------
// Everything of a Lanczos step except the operator application, in one single-CTA launch: both
// Gram-Schmidt passes against the nb leading basis vectors, the norm, the next basis vector and its
// scaled copy, and -- at check steps -- the projected eigenproblem, whose verdict is latched in
// state[1] so that the launches already queued behind it (matvec and tail both test the flag) fall
// through.  The host therefore synchronises once per chunk of steps instead of once per check.
// state: [0] breakdown step, [1] done, [2] step at which done was raised.
constexpr int kFusedMax = 4096;

__global__ void __launch_bounds__(kOneCta)
lanczos_tail(int m, int j, int nb, int hj, int check, const double *basis, const double *__restrict__ w_in,
             const double *__restrict__ isd, double *alpha, double *beta, double *next, double *__restrict__ z,
             int32_t *state, double *coef, double *ritz) {
    specdev::lanczos_tail_body(m, j, nb, hj, check, basis, w_in, isd, alpha, beta, next, z, state, coef, ritz);
}

// y = sum_{k=1..j} coef[k] v_k, normalised (`basis` points at v_0, the row before v_1);
// z = isd .* y.  One CTA.
__global__ void __launch_bounds__(kOneCta)
ritz_vector(int m, int j, const double *__restrict__ basis, const double *__restrict__ coef,
            const double *__restrict__ isd, double *__restrict__ y, double *__restrict__ z) {
    specdev::ritz_vector_body(m, j, basis, coef, isd, y, z);
}

// out[0] = | Ny - theta y |, out[1] = y . Ny   (Ny given).  One CTA.
__global__ void __launch_bounds__(kOneCta)
true_residual(int m, const double *__restrict__ y, const double *__restrict__ Ny, const double *__restrict__ ritz,
              double *__restrict__ out) {
    specdev::true_residual_body(m, y, Ny, ritz, out);
}

// ---- embedding, sign flip, exact 1-D 2-means --------------------------------------------------
// u = y .* isd is the Fiedler coordinate sklearn clusters (_spectral_embedding.py:378-381); its sign is
// fixed so that the entry of largest magnitude is positive (extmath.py:1283-1286).  The 2-means optimum
// in one dimension is a threshold on the sorted values: sort, prefix sums, best split.
// result: [0] margin, [1] lower centroid, [2] upper centroid, [3] size of the upper part,
//         [4] number of Lloyd-stable splits, [5] best other stable split's score / the optimum's
template <bool kShared>
__global__ void __launch_bounds__(kOneCta)
two_means_1d(int m, int P, const double *__restrict__ y, const double *__restrict__ isd, double *__restrict__ u,
             double *__restrict__ sorted_g, int32_t *__restrict__ side, double *__restrict__ result) {
    specdev::two_means_1d_body<kShared>(m, P, y, isd, u, sorted_g, side, result);
}

template <int kStage>
__global__ void __launch_bounds__(kOneCta)
two_means_staged(int m, int P, const double *__restrict__ y, const double *__restrict__ isd, double *__restrict__ u,
                 double *__restrict__ sorted_g, int32_t *__restrict__ side, double *__restrict__ result) {
    specdev::two_means_1d_body<false, kStage>(m, P, y, isd, u, sorted_g, side, result);
}

// ---- sort of more keys than one CTA's shared memory holds: bitonic network over many CTAs ----------------------------
// Tiles of kSortTile keys are sorted / merged in shared memory (every compare distance below the tile size); the
// larger distances are one launch each over all pairs.  Ascending; P is a power of two >= 2 * kSortTile.
constexpr int kSortTile = 4096;

// all stages k = 2 .. kSortTile of the network on one tile (first = 1), or the distances jmax .. 1 of stage k
__global__ void __launch_bounds__(1024)
sort_tile(double *__restrict__ keys, int first, int k_global, int jmax) {
    __shared__ double tile[kSortTile];
    const int base = blockIdx.x * kSortTile, tid = threadIdx.x;
    for (int i = tid; i < kSortTile; i += 1024) tile[i] = keys[base + i];
    __syncthreads();
    for (int k = first ? 2 : k_global; k <= (first ? kSortTile : k_global); k <<= 1) {
        for (int jj = first ? k >> 1 : jmax; jj > 0; jj >>= 1) {
            for (int i = tid; i < kSortTile; i += 1024) {
                const int partner = i ^ jj;
                if (partner > i) {
                    const double x0 = tile[i], x1 = tile[partner];
                    const bool up = ((base + i) & k) == 0;
                    if ((x0 > x1) == up) {
                        tile[i] = x1;
                        tile[partner] = x0;
                    }
                }
            }
            __syncthreads();
        }
    }
    for (int i = tid; i < kSortTile; i += 1024) keys[base + i] = tile[i];
}

// one compare distance j >= kSortTile of stage k over the whole array
__global__ void sort_far(double *__restrict__ keys, int P, int k, int j) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;  // pair index
    if (t >= P / 2) return;
    const int i = ((t / j) * 2 * j) + (t % j);  // the lower element of the pair
    const int partner = i + j;
    const double x0 = keys[i], x1 = keys[partner];
    const bool up = (i & k) == 0;
    if ((x0 > x1) == up) {
        keys[i] = x1;
        keys[partner] = x0;
    }
}

int sort_keys(scs_ctx *ctx, double *keys, int P) {
    sort_tile<<<P / kSortTile, 1024, 0, ctx->stream>>>(keys, 1, 0, 0);
    SCS_LAUNCHED(ctx, "sort_tile");
    for (int k = 2 * kSortTile; k <= P; k <<= 1) {
        for (int j = k >> 1; j >= kSortTile; j >>= 1) {
            sort_far<<<ceil_div(P / 2, 256), 256, 0, ctx->stream>>>(keys, P, k, j);
            SCS_LAUNCHED(ctx, "sort_far");
        }
        sort_tile<<<P / kSortTile, 1024, 0, ctx->stream>>>(keys, 0, k, kSortTile >> 1);
        SCS_LAUNCHED(ctx, "sort_tile");
    }
    return SCS_OK;
}

__global__ void trivial_pair(int32_t *side) {
    side[0] = 0;
    side[1] = 1;
}

int next_pow2(int x) {
    int p = 1;
    while (p < x) p <<= 1;
    return p;
}

}  // namespace

int normalized_matvec(scs_ctx *ctx, int m, const double *W, const double *isd, const double *x, double *y) {
    if (m <= 0 || !W || !isd || !x || !y) return fail(ctx, SCS_ERR_INVALID, "normalized_matvec: bad argument");
    double *z;
    int rc;
    if ((rc = reserve_as(ctx, SLOT_UVEC, static_cast<size_t>(m), &z))) return rc;
    scale_vector<<<ceil_div(m, 256), 256, 0, ctx->stream>>>(m, isd, x, z);
    SCS_LAUNCHED(ctx, "scale_vector");
    return launch_matvec_single(ctx, m, W, isd, z, y, nullptr);
}

namespace {

struct LanczosOutcome {
    double theta1 = 0.0, theta2 = 0.0, estimate = 0.0;
    int steps = 0;        // size of the projected problem that produced the pair
    bool converged = false;
    bool invariant = false;  // stopped on a breakdown: the Krylov space is an invariant subspace
    int matvecs = 0;
    int restarts = 0;
};

struct LanczosBuffers {
    double *isd, *basis, *w, *z, *coef, *h1, *h2, *alpha, *beta, *ritz;
    int32_t *state;
    double *pin;
};

// Largest eigenpair of N = D^-1/2 W D^-1/2 on the orthogonal complement of the first `ndefl` rows of
// `basis`.  Lanczos vectors go to rows ndefl, ndefl+1, ...; the Ritz vector to `y` (and isd .* y to z).
int lanczos_largest(scs_ctx *ctx, int m, const double *W, const LanczosBuffers &b, int ndefl, uint64_t seed,
                    double *y, LanczosOutcome *out, RowBlock rows) {
    const int dim = m - ndefl;  // dimension of the deflated space
    const int jmax = dim < kMaxBasis ? dim : kMaxBasis;
    const int vec_blocks = ceil_div(m, kVecThreads);
    double *v0 = b.basis + static_cast<size_t>(ndefl - 1) * m;  // v_k lives at v0 + k m
    double *w = b.w;  // the vector being orthogonalised: b.w, or the window buffer a sharded matvec filled
    int rc;
    int jdone = 0;
    const bool fused = m <= kFusedMax;
    if (fused && !ctx->tail_configured) {
        SCS_CUDA(ctx, cudaFuncSetAttribute(lanczos_tail, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           static_cast<int>((kFusedMax + 6 * (kMaxBasis + 8)) * sizeof(double))));
        ctx->tail_configured = true;
    }
    const size_t tail_smem = (static_cast<size_t>(m) + 6 * (kMaxBasis + 8)) * sizeof(double);
    // everything of step j but the matvec: one CTA up to kFusedMax, one cluster above
    auto step_tail = [&](int j, int check) -> int {
        const int nb = j == 0 ? ndefl : ndefl + j;
        const int hj = j == 0 ? 0 : ndefl - 1 + j;
        double *next = v0 + static_cast<size_t>(j + 1) * m;
        if (fused) {
            lanczos_tail<<<1, kOneCta, tail_smem, ctx->stream>>>(m, j, nb, hj, check, b.basis, w, b.isd, b.alpha, b.beta,
                                                                next, b.z, b.state, b.coef, b.ritz);
            SCS_LAUNCHED(ctx, "lanczos_tail");
        } else {
            lanczos_step<<<kStepCluster, kVecThreads, kStepSmem, ctx->stream>>>(m, j, nb, hj, check, b.basis, w, b.isd,
                                                                               b.h1, b.h2, b.alpha, b.beta, next, b.z,
                                                                               b.state, b.coef, b.ritz);
            SCS_LAUNCHED(ctx, "lanczos_step");
        }
        return SCS_OK;
    };
    for (int attempt = 0; attempt <= kMaxRestarts && !out->converged; ++attempt) {
        w = b.w;
        if (attempt == 0) {
            random_start<<<vec_blocks, kVecThreads, 0, ctx->stream>>>(m, seed, b.w);
            SCS_LAUNCHED(ctx, "random_start");
        } else {
            // explicit restart from the current Ritz vector
            SCS_CUDA(ctx, cudaMemcpyAsync(b.w, y, sizeof(double) * m, cudaMemcpyDeviceToDevice, ctx->stream));
            out->restarts = attempt;
        }
        SCS_CUDA(ctx, cudaMemsetAsync(b.state, 0, 4 * sizeof(int32_t), ctx->stream));
        if ((rc = step_tail(0, 0))) return rc;
        // steps are queued a chunk at a time; the tail of a check step latches convergence on the
        // device and everything queued behind it falls through
        int j = 1;
        int attempt_matvecs = 0;
        bool done = false;
        while (j <= jmax && !done) {
            const int chunk_end = std::min(jmax, j == 1 ? 16 : j + 3);  // chunks end on check steps
            for (; j <= chunk_end; ++j) {
                if ((rc = launch_matvec(ctx, m, W, b.isd, b.z, &w, b.state + 1, rows))) return rc;
                if ((rc = step_tail(j, j == jmax || (j % 4) == 0))) return rc;
            }
            SCS_CUDA(ctx, cudaMemcpyAsync(b.pin, b.ritz, 6 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
            SCS_CUDA(ctx, cudaMemcpyAsync(b.pin + 6, b.state, 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
            SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            const int32_t *st = reinterpret_cast<const int32_t *>(b.pin + 6);
            out->theta1 = b.pin[0];
            out->theta2 = b.pin[1];
            out->estimate = b.pin[2];
            out->steps = static_cast<int>(b.pin[4]);
            jdone = static_cast<int>(b.pin[5]);  // the step of the last check that ran
            if (st[1]) {
                done = true;
                out->converged = true;
                out->invariant = b.pin[3] <= kBreakdown;
                attempt_matvecs = st[2];  // steps actually applied before the flag went up
            } else {
                attempt_matvecs = chunk_end;
            }
        }
        out->matvecs += attempt_matvecs;
        // Ritz vector of the current basis (also the restart vector); coefficients past a breakdown are 0
        ritz_vector<<<1, kOneCta, (jdone + 1) * sizeof(double), ctx->stream>>>(m, jdone, v0, b.coef, b.isd, y, b.z);
        SCS_LAUNCHED(ctx, "ritz_vector");
    }
    return SCS_OK;
}

}  // namespace

int spectral_bipartition(scs_ctx *ctx, int m, const double *W, const double *degree, uint64_t seed, int32_t *side,
                         scs_node_stats *stats, RowBlock rows) {
    if (rows.sharded() && !degree) return fail(ctx, SCS_ERR_INVALID, "sharded spectral step needs the degrees");
    if (m < 2 || !W || !side || !stats) return fail(ctx, SCS_ERR_INVALID, "spectral_bipartition: bad argument");
    int rc;
    if (m == 2) {
        // sklearn falls back to a dense eigh (arpack.py:1691-1707); two vertices always separate
        trivial_pair<<<1, 1, 0, ctx->stream>>>(side);
        SCS_LAUNCHED(ctx, "trivial_pair");
        stats->solver = 1;
        stats->eig[1] = 2.0;  // L = [[1,-1],[-1,1]] whatever the weight
        stats->residual = 0.0;
        stats->margin = 0.5;
        return SCS_OK;
    }
    const int jcap = m - 1 < kMaxBasis ? m - 1 : kMaxBasis;
    LanczosBuffers b;
    double *tri, *embed, *sorted, *deg_own, *work;
    int32_t *flags;
    if ((rc = reserve_as(ctx, SLOT_ISD, static_cast<size_t>(m), &b.isd))) return rc;
    if ((rc = reserve_as(ctx, SLOT_BASIS, static_cast<size_t>(jcap + 3) * m, &b.basis))) return rc;
    if ((rc = reserve_as(ctx, SLOT_WORK, 3 * static_cast<size_t>(m), &work))) return rc;
    if ((rc = reserve_as(ctx, SLOT_UVEC, static_cast<size_t>(m), &b.z))) return rc;
    if ((rc = reserve_as(ctx, SLOT_COEF, 3 * static_cast<size_t>(kMaxBasis + 8), &b.coef))) return rc;
    if ((rc = reserve_as(ctx, SLOT_TRIDIAG, 2 * static_cast<size_t>(kMaxBasis + 8), &tri))) return rc;
    if ((rc = reserve_as(ctx, SLOT_RITZ, 32, &b.ritz))) return rc;
    if ((rc = reserve_as(ctx, SLOT_EMBED, static_cast<size_t>(m), &embed))) return rc;
    const int P = next_pow2(m);
    if ((rc = reserve_as(ctx, SLOT_SORTED, static_cast<size_t>(P), &sorted))) return rc;
    if ((rc = reserve_as(ctx, SLOT_SPEC_SCALARS, 16, &flags))) return rc;
    b.h1 = b.coef + (kMaxBasis + 8);
    b.h2 = b.h1 + (kMaxBasis + 8);
    b.alpha = tri;
    b.beta = tri + (kMaxBasis + 8);
    b.w = work;
    b.state = flags + 4;
    double *yvec = work + m, *y2 = work + 2 * static_cast<size_t>(m);
    void *pin_v;
    if ((rc = reserve_pinned(ctx, 256, &pin_v))) return rc;
    b.pin = static_cast<double *>(pin_v);
    double *pin = b.pin;

    SCS_CUDA(ctx, cudaMemsetAsync(flags, 0, 16 * sizeof(int32_t), ctx->stream));
    if (!degree) {
        if ((rc = reserve_as(ctx, SLOT_DEGREE_C, static_cast<size_t>(m), &deg_own))) return rc;
        row_sums<<<ceil_div(static_cast<int64_t>(m) * 32, 256), 256, 0, ctx->stream>>>(m, W, deg_own);
        SCS_LAUNCHED(ctx, "row_sums");
        degree = deg_own;
    }
    prepare_scaling<<<1, kOneCta, 0, ctx->stream>>>(m, degree, b.isd, b.basis, flags);
    SCS_LAUNCHED(ctx, "prepare_scaling");

    stats->solver = 3;
    LanczosOutcome first;
    const auto t_lanczos = std::chrono::steady_clock::now();
    if ((rc = lanczos_largest(ctx, m, W, b, 1, seed, yvec, &first, rows))) return rc;
    ctx->stage_seconds[5] += std::chrono::duration<double>(std::chrono::steady_clock::now() - t_lanczos).count();
    stats->matvecs = first.matvecs;
    stats->restarts = first.restarts;

    // true residual of the accepted pair: one more operator application (z = isd .* y is current)
    double *Ny = b.w;
    if ((rc = launch_matvec(ctx, m, W, b.isd, b.z, &Ny, nullptr, rows))) return rc;
    stats->matvecs += 1;
    true_residual<<<1, kOneCta, 0, ctx->stream>>>(m, yvec, Ny, b.ritz, b.ritz + 8);
    SCS_LAUNCHED(ctx, "true_residual");
    SCS_CUDA(ctx, cudaMemcpyAsync(pin + 8, b.ritz + 8, 2 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));

    // The second Ritz value of the same Krylov space only bounds the next eigenvalue from below.  If the
    // space closed early (fewer than m - 1 steps), an eigenvalue of N is repeated -- possibly the Fiedler
    // one.  Settle it with a second run deflated by the Fiedler vector as well.
    double theta_next = first.theta2;
    if (first.invariant && first.steps < m - 1 && m >= 3) {
        SCS_CUDA(ctx, cudaMemcpyAsync(b.basis + m, yvec, sizeof(double) * m, cudaMemcpyDeviceToDevice, ctx->stream));
        LanczosOutcome second;
        b.ritz += 16;  // keep the first pair's scalars
        rc = lanczos_largest(ctx, m, W, b, 2, seed + 0x5bd1e995u, y2, &second, rows);
        b.ritz -= 16;
        if (rc) return rc;
        stats->matvecs += second.matvecs;
        theta_next = second.theta1;
    }

    if (P <= 8192) {
        auto kernel = two_means_1d<true>;
        const size_t smem = static_cast<size_t>(P) * sizeof(double);
        if (!ctx->kmeans_configured) {
            SCS_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 8192 * 8));
            ctx->kmeans_configured = true;
        }
        kernel<<<1, kOneCta, smem, ctx->stream>>>(m, P, yvec, b.isd, embed, sorted, side, b.ritz + 12);
    } else {
        // more keys than one CTA sorts in shared memory: embedding and keys, a sort over many CTAs, then the rest
        two_means_staged<1><<<1, kOneCta, 0, ctx->stream>>>(m, P, yvec, b.isd, embed, sorted, side, b.ritz + 12);
        SCS_LAUNCHED(ctx, "two_means_staged");
        if ((rc = sort_keys(ctx, sorted, P))) return rc;
        two_means_staged<2><<<1, kOneCta, 0, ctx->stream>>>(m, P, yvec, b.isd, embed, sorted, side, b.ritz + 12);
    }
    SCS_LAUNCHED(ctx, "two_means_1d");
    SCS_CUDA(ctx, cudaMemcpyAsync(pin + 12, b.ritz + 12, 6 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    SCS_CUDA(ctx, cudaMemcpyAsync(pin + 20, flags, 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    stats->eig[0] = 0.0;
    stats->eig[1] = 1.0 - first.theta1;
    stats->eig[2] = 1.0 - theta_next;
    stats->residual = pin[8];
    stats->margin = pin[12];
    const int32_t bad_degree = reinterpret_cast<const int32_t *>(pin + 20)[0];
    stats->kmeans_stable_splits = static_cast<int32_t>(pin[16]);
    stats->kmeans_runner_up = pin[17];
    stats->tie_flag = 0;
    if (!std::isnan(theta_next) && (first.theta1 - theta_next) < kGapTie) stats->tie_flag |= 1;
    if (!(stats->margin >= kMarginTie)) stats->tie_flag |= 2;
    if (!first.converged) stats->tie_flag |= 4;  // accepted at the restart limit: see stats->residual
    if (bad_degree) stats->tie_flag |= 8;        // negative / non-finite degree: sklearn's result is NaN-driven
    if (stats->kmeans_stable_splits > 1) stats->tie_flag |= 16;  // k-means has several local optima
    return SCS_OK;
}

}  // namespace scs
