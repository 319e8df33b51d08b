// Internal definitions shared by the translation units of libscs_b200.so.
#pragma once

#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "scs_b200.h"

namespace scs {

constexpr int kMediumMaxDefault = 4096;

// A grow-only device allocation; a context keeps one per purpose so steady-state recursion
// nodes allocate nothing.
struct DeviceBuffer {
    void *ptr = nullptr;
    size_t bytes = 0;
};

enum Slot : int {
    // leaf tours copied in by the host-facing call
    SLOT_TOUR_OFFSETS = 0,
    SLOT_TOUR_TAXON,
    SLOT_TOUR_DEPTH,
    SLOT_TOUR_VAL,
    SLOT_TOUR_ROOT,
    SLOT_TOUR_WEIGHT,
    // proper cluster graph
    SLOT_W,
    SLOT_WC,
    SLOT_OCC,
    SLOT_ADJ_BITS,
    SLOT_MAX_BITS,
    SLOT_DEGREE,
    SLOT_DEGREE_C,
    SLOT_LEAF_TREE,
    SLOT_ROW_PTR,
    SLOT_CURSOR,
    SLOT_INV,
    SLOT_INV_SORTED,
    SLOT_DEGREE_PART,
    SLOT_LINKS,
    SLOT_BUCKET_COUNT,  // per-leaf staircases of the graph build (LeafStairs)
    SLOT_START16,       // per leaf: where each warp's share of the tree starts in triangle mode
    SLOT_BUCKET_PTR,
    SLOT_ENTRIES,
    // components / contraction
    SLOT_UF_PARENT,
    SLOT_LABEL,
    SLOT_LABEL2,
    SLOT_GROUP,
    SLOT_GROUP_PTR,
    SLOT_GROUP_MEMBERS,
    SLOT_SCALARS,
    SLOT_PART,
    // spectral
    SLOT_ISD,
    SLOT_UVEC,
    SLOT_BASIS,
    SLOT_WORK,
    SLOT_COEF,
    SLOT_TRIDIAG,
    SLOT_RITZ,
    SLOT_EMBED,
    SLOT_SORTED,
    SLOT_SIDE,
    SLOT_SPEC_SCALARS,
    SLOT_L2_FLUSH,
    SLOT_NODE_STATS,
    // batched medium-node path (medium.cu)
    SLOT_MED_NODES,
    SLOT_MED_ROW_NODE,
    SLOT_MED_TREE_NODE,
    SLOT_MED_STATE,
    SLOT_MED_VEC,
    SLOT_MED_SMALL,
    SLOT_MED_STAGE,
    SLOT_SCAN_SUMS,
    SLOT_COUNT
};

constexpr int kMaxPeers = 16;  // GPUs that can share one recursion node (shard.cu)

// Where the pieces of a rank's exchange window live (byte offsets; the same on every rank).
struct ShardLayout {
    size_t vec[2] = {0, 0};  // double-buffered all-gather target of the sharded matvec, n_max doubles each
    size_t degree = 0, degree_c = 0;  // n_max doubles each
    size_t adj_bits = 0, max_bits = 0;  // n_max * words(n_max) uint32 each
    size_t W = 0;  // this rank's row block of W: rows_per_rank(n_max) * n_max doubles
    size_t total = 0;
};

// Row-sharded recursion nodes over the GPUs of one box (shard.cu / shard.cuh).
struct ShardState {
    bool connected = false;  // peers' windows are mapped
    bool engaged = false;    // the caller guarantees that every rank issues the same node calls
    int rank = 0, world = 1;
    int n_max = 0;           // largest node the window was sized for
    int min_n = 4096;        // nodes with fewer taxa stay on one GPU
    unsigned long long epoch = 0;  // synchronisation points issued so far
    int parity = 0;          // which vec buffer the next sharded matvec fills
    double timeout_s = 20.0;  // bound on every device-side wait
    unsigned char *window = nullptr;  // own window (cudaMalloc)
    unsigned char *peer[kMaxPeers] = {};  // mapped windows, peer[rank] == window
    bool opened[kMaxPeers] = {};  // mapped with cudaIpcOpenMemHandle by this context
    ShardLayout layout;
    int64_t nodes = 0;  // recursion nodes that took the sharded path
};

// Rows [row0, row1) of a row-sharded matrix live on this rank; row1 < 0 means "not sharded".
struct RowBlock {
    int row0 = 0, row1 = -1;
    // graph build of a row block: every row computes only the cyclic half window of columns after its own (each
    // pair of the node once, over all ranks); the caller completes the rows from the peers' blocks
    // (pcg_fetch_transposed), the bit matrices (pcg_symmetrize_bits) and sums them (pcg_degree_block)
    bool half_window = false;
    bool sharded() const { return row1 >= 0; }
};

// One recursion node of a batch of medium-sized nodes (medium.cu): where its rows, trees and matrices live in
// the batch's concatenated buffers.  Filled on the host, read-only on the device.
struct MedNode {
    int32_t n, words;         // vertices; 32-bit words per adjacency-bit row
    int32_t row_base;         // first row of the node in the batch's global row space
    int32_t tree_begin, tree_end;  // its trees in the batch's tree arrays
    int32_t jcap;             // Lanczos vectors its basis block can hold (min(n - 1, kMaxBasis))
    int32_t blk_base, pad0;   // first 32-row block of the node among the batch's row blocks (sum of ceil(n / 32))
    int64_t w_off;            // first element of its n x n block in the W (and Wc) buffer
    int64_t bit_off;          // first word of its bit rows in the adjacency / max-graph buffers
    int64_t basis_off;        // first element of its (jcap + 3) x n basis block
    int64_t part_off;         // where its n partition labels go in the caller's part array
    uint64_t seed;            // picks the Lanczos start vector
};

inline int shard_rows_per_rank(int n, int world) { return (n + world - 1) / world; }
inline RowBlock shard_block(int n, int rank, int world) {
    const int per = shard_rows_per_rank(n, world);
    RowBlock b;
    b.row0 = rank * per < n ? rank * per : n;
    b.row1 = b.row0 + per < n ? b.row0 + per : n;
    return b;
}

}  // namespace scs

struct scs_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sm_count = 148;
    size_t smem_optin = 0;
    size_t smem_per_sm = 0;
    int64_t launches = 0;
    std::string last_error;
    scs::DeviceBuffer slots[scs::SLOT_COUNT];
    void *pinned = nullptr;  // host staging for small results
    size_t pinned_bytes = 0;
    void *pinned_io = nullptr;  // host staging for the tours of scs_node_split_host
    size_t pinned_io_bytes = 0;
    int64_t h2d_bytes = 0;  // bytes copied by the *_host entry points
    int64_t d2h_bytes = 0;
    // optional per-launch timing of the two heavy kernels (bench.py's roofline figures)
    bool profile_on = false;
    struct ProfileRecord {
        cudaEvent_t start, stop;
        int kind;
        double bytes, units;
    };
    std::vector<ProfileRecord> profile;
    int flush_value = 0;
    double stage_seconds[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // host wall clock per stage of the staged node path
    std::vector<scs_ctx *> workers;  // extra contexts on the same GPU for concurrent staged nodes
    bool small_configured = false;
    bool batch_configured = false;
    bool tail_configured = false;
    bool rows_configured[32] = {};
    bool mirror_configured = false;
    bool contract_configured = false;
    bool kmeans_configured = false;
    bool medium_configured = false;
    bool device_forest = true;  // scs_supertree_build on one GPU keeps the source trees on the device (devdriver.cu)
    int medium_limit = scs::kMediumMaxDefault;  // nodes up to this size (and above small_limit) go through the batched path
    bool wide_entries = false;  // graph build: 8-byte bucket entries even where 4 bytes would do (tests)
    bool full_rows = false;     // graph build: every row CTA visits all its pairs (no triangle + mirror; tests, A/B timing)
    // nodes up to this size take the one-CTA path (0 disables it; capacity kSmallNode = 64).  32 by measurement: one CTA
    // needs ~3 ms for a 64-taxon node covered by hundreds of trees (tree loop + Jacobi sweeps), which made the small
    // batch the critical path of every wave; up to 32 taxa it stays below 1 ms and the medium batch takes the rest
    int small_limit = 32;
    double pending_units = 0.0;  // leaf-pair visits of the node being built (set by host entry points)
    cudaEvent_t timer_start = nullptr, timer_stop = nullptr;
    // shape of the node most recently processed by scs_node_split_host
    int last_n = 0;
    int last_m = 0;
    scs::ShardState shard;
    // device buffers of the recursion driver that survive from one build to the next (devdriver.cu): a build then
    // allocates nothing -- fresh gigabyte-sized allocations stalled single waves by hundreds of milliseconds
    void *driver_cache = nullptr;
    void (*driver_cache_release)(scs_ctx *, void *) = nullptr;
};

namespace scs {

int fail(scs_ctx *ctx, int status, const char *what, cudaError_t err = cudaSuccess);

#define SCS_CUDA(ctx, call)                                                   \
    do {                                                                      \
        cudaError_t err__ = (call);                                           \
        if (err__ != cudaSuccess) return scs::fail(ctx, SCS_ERR_CUDA, #call, err__); \
    } while (0)

// Check the launch that was just issued and count it.
#define SCS_LAUNCHED(ctx, name)                                               \
    do {                                                                      \
        cudaError_t err__ = cudaGetLastError();                               \
        if (err__ != cudaSuccess) return scs::fail(ctx, SCS_ERR_CUDA, name, err__); \
        (ctx)->launches += 1;                                                 \
    } while (0)

// Device memory for `slot`, at least `bytes` large (contents undefined after growth).
int reserve(scs_ctx *ctx, Slot slot, size_t bytes, void **out);

template <typename T>
inline int reserve_as(scs_ctx *ctx, Slot slot, size_t count, T **out) {
    void *p = nullptr;
    int rc = reserve(ctx, slot, count * sizeof(T), &p);
    *out = static_cast<T *>(p);
    return rc;
}

int reserve_pinned(scs_ctx *ctx, size_t bytes, void **out);

enum ProfileKind : int { PROFILE_MATVEC = 0, PROFILE_PCG_ROWS = 1, PROFILE_KINDS = 2 };
constexpr int kSmallNode = 64;  // recursion nodes up to this many vertices take the one-CTA path (small.cu)
constexpr int kSmallCap32 = 32;  // ... those up to this many the smaller-capacity instance of it
constexpr int kSmallMaxTrees = 65535;  // ... if they have at most this many source trees (16-bit co-occurrence counts)
// the per-launch roofline timers cover the launches whose matrix exceeds the 126 MB L2 (8 n^2 bytes > L2 from
// n = 3969); smaller matrices stay L2-resident across the matvecs of a Lanczos run: no HBM roofline there
constexpr int kProfileMinSize = 4096;

// Bracket the launch that follows / preceded with events when profiling is on.
void profile_begin(scs_ctx *ctx, int kind, double bytes, double units);
void profile_end(scs_ctx *ctx);

inline int ceil_div(int64_t a, int64_t b) { return static_cast<int>((a + b - 1) / b); }

// out[i] = in[0] + ... + in[i-1] for i in [0, n]  (out has n + 1 entries)
int exclusive_scan(scs_ctx *ctx, int n, const int32_t *in, int32_t *out);

// monotone map double -> uint64 for max-reductions with integer atomics (0 is below every real
// number: used for "no edge")
#ifdef __CUDACC__
__device__ __forceinline__ unsigned long long order_key(double x) {
    const unsigned long long sign = 0x8000000000000000ull;
    unsigned long long b = static_cast<unsigned long long>(__double_as_longlong(x));
    return (b & sign) ? ~b : (b | sign);
}
__device__ __forceinline__ double order_value(unsigned long long k) {
    const unsigned long long sign = 0x8000000000000000ull;
    unsigned long long b = (k & sign) ? (k & ~sign) : ~k;
    return __longlong_as_double(static_cast<long long>(b));
}
#endif

// Large buffers of `ctx` sized for a node of n taxa, T trees, L leaves (context.cu).
int prewarm_node(scs_ctx *ctx, int n, int T, int64_t L);

// Make sure ctx->workers holds at least `count - 1` extra contexts (the main context is worker 0).
int ensure_workers(scs_ctx *ctx, int count);

// ---- stage entry points implemented in the other translation units ------------------------
// `rows`: build only those rows (W / C then point at the row block: row a is at (a - row0) * n; the
// bit matrices and degree stay full-size and are indexed by the global row).
int pcg_build(scs_ctx *ctx, int n, int T, int64_t L, const int64_t *leaf_offsets,
              const int32_t *leaf_taxon, const int32_t *adj_depth, const double *adj_val,
              const int32_t *root_depth, const double *tree_weight, double *W, int32_t *C,
              int32_t *occ, uint32_t *adj_bits, uint32_t *max_bits, double *degree, RowBlock rows = RowBlock());

// Completion of a half-window row block (see RowBlock): peer_W[r] = rank r's row block (rows [r * rows_per_rank, ...),
// row stride n), all of them finished with their own halves; the bit matrices are the full n x n ones every rank
// holds after the exchange of the rows.
int pcg_fetch_transposed(scs_ctx *ctx, int n, RowBlock rows, int rows_per_rank, int world, const double *const *peer_W,
                         double *W_block);
int pcg_symmetrize_bits(scs_ctx *ctx, int n, uint32_t *adj_bits, uint32_t *max_bits);
int pcg_degree_block(scs_ctx *ctx, int n, int T, RowBlock rows, const double *W_block, double *degree);

int components(scs_ctx *ctx, int n, const uint32_t *bits, int32_t *label, int32_t *n_components_host);

int components_async(scs_ctx *ctx, int n, const uint32_t *bits, int32_t *label, int32_t *count_dev);

// The same labels from the node's leaf tours, without its graph; *bad_dev is raised for a malformed tour.
int tour_components_async(scs_ctx *ctx, int n, int T, int64_t L, const int64_t *leaf_offsets,
                          const int32_t *leaf_taxon, const int32_t *adj_depth, const int32_t *root_depth,
                          int32_t *label, int32_t *count_dev, int32_t *bad_dev);

int contract(scs_ctx *ctx, int n, const double *W, const uint32_t *adj_bits, const uint32_t *max_bits,
             int32_t *group, int32_t *m_host, double *Wc, double *degree_c);
// `rows` (sharded): only contracted rows [row0, row1) are produced, into the row block Wc; W is then read
// through the peers' windows (row u of W lives on rank u / rows_per_rank(n)).
int contract_with_labels(scs_ctx *ctx, int n, const double *W, const uint32_t *adj_bits, const int32_t *label, int m,
                         int32_t *group, double *Wc, double *degree_c, RowBlock rows = RowBlock());

// `rows` (sharded): W is this rank's row block; every operator application is the fused
// matvec + all-gather over the peers' windows, everything else is replicated on every rank.
int spectral_bipartition(scs_ctx *ctx, int m, const double *W, const double *degree, uint64_t seed,
                         int32_t *side, scs_node_stats *stats_host, RowBlock rows = RowBlock());

int normalized_matvec(scs_ctx *ctx, int m, const double *W, const double *isd, const double *x, double *y);

// Graph build of a batch of nodes in one set of launches (pcg.cu): R rows in all, T trees, L leaves; the tours are
// concatenated with absolute leaf offsets; W / bit matrices are addressed through the node table.
int pcg_build_batch(scs_ctx *ctx, int B, int blocks, int R, int T, int64_t L, int max_n, int max_trees, const MedNode *nodes_dev,
                    const int32_t *tree_node, const int32_t *row_node, const int64_t *leaf_offsets,
                    const int32_t *leaf_taxon, const int32_t *adj_depth, const double *adj_val,
                    const int32_t *root_depth, const double *tree_weight, double *W, int32_t *occ, uint32_t *adj_bits,
                    uint32_t *max_bits, double *degree, int32_t *bad_dev);

constexpr int kMediumMax = kMediumMaxDefault;  // recursion nodes up to this many vertices can go through the batched path

// A batch of recursion nodes (kSmallNode < n <= kMediumMax is what the driver sends), every stage one launch over
// all of them (medium.cu).  Tours: concatenated, node b owns trees [tree_begin[b], tree_end[b]) (ascending, disjoint;
// trees in between belong to nobody and are skipped) and their leaves; leaf_offsets[T + 1] absolute; all tour
// pointers are device pointers.  part_dev receives the labels of node b at part_off[b]; stats_host[b] its record.
// needs_rerun[b] is set when the node has to go through scs_node_split_* instead (eigensolver restart or a
// repeated-eigenvalue check: rare).
int medium_batch(scs_ctx *ctx, int B, const int32_t *node_n, const int32_t *tree_begin, const int32_t *tree_end,
                 const int64_t *part_off, const uint64_t *seeds, int T, int64_t L, const int64_t *leaf_offsets, const int32_t *leaf_taxon,
                 const int32_t *adj_depth, const double *adj_val, const int32_t *root_depth, const double *tree_weight,
                 int contract_edges, int32_t *part_dev, scs_node_stats *stats_host, uint8_t *needs_rerun);

// Components, contraction and the spectral split of a graph of <= kSmallNode vertices in one launch;
// part / out_dev / group_out / Wc_out are device pointers (the last two may be null).
int small_node(scs_ctx *ctx, int n, int contract_edges, const double *W, const uint32_t *adj_bits,
               const uint32_t *max_bits, int32_t *part, scs_node_stats *out_dev, int32_t *group_out,
               double *Wc_out);

// Launch order of a batch of small nodes (host arrays): the nodes of at most kSmallCap32 vertices first, each group
// heaviest first (n^2 x trees) so that no heavy node starts in the last round of CTAs.  Returns the size of the first
// group.
int small_order(int num_nodes, const scs_small_node *nodes, int32_t *order);

// A batch of small nodes, one CTA each, graph build included; all pointers are device pointers.  order_dev (from
// small_order, num_cap32 its return value) is the launch order: the first num_cap32 nodes of it run on the
// 32-capacity kernel, the rest on the 64-capacity one.  order_dev null: every node on the 64-capacity kernel, in
// descriptor order.  Stats and labels land at each node's own slot either way.
// absolute_offsets: leaf_offsets[tree_base + t] is the absolute tour position of tree t of a node (the device forest's
// layout); otherwise node b reads leaf_offsets[tree_base + b + t], relative to its leaf_base (scs_small_node's layout).
int small_batch(scs_ctx *ctx, int num_nodes, const scs_small_node *nodes_dev, const int32_t *order_dev, int num_cap32,
                const int64_t *leaf_offsets, const int32_t *leaf_taxon, const int32_t *adj_depth, const double *adj_val,
                const int32_t *root_depth, const double *tree_weight, int contract_edges, int32_t *part_dev,
                scs_node_stats *stats_dev, int32_t *bad_dev, int absolute_offsets = 0);

// SM cycles the batched small-node kernel spent in its graph build / in everything after it, summed over CTAs.
int small_cycles(scs_ctx *ctx, unsigned long long *out2, int reset);

// One recursion node on device-resident tours.  part_dev[n] receives the component index or side;
// if part_host is not null the result is also copied there before the function returns.
// tour_components (the recursion drivers): a node above the small limit is first split into the components
// of its tours, and a disconnected one returns without building its graph.  Off, the graph is always built,
// so that scs_node_last_buffers shows W and the bits of every node.
int node_split(scs_ctx *ctx, int n, int T, int64_t L, const int64_t *leaf_offsets, const int32_t *leaf_taxon,
               const int32_t *adj_depth, const double *adj_val, const int32_t *root_depth,
               const double *tree_weight, int contract_edges, uint64_t seed, int32_t *part_dev,
               int32_t *part_host, scs_node_stats *stats, bool tour_components = false);

// scs_node_split_host with the choice above (driver.cu's host-forest recursion passes true).
int node_split_host(scs_ctx *ctx, int n, int T, int64_t L, const int64_t *leaf_offsets, const int32_t *leaf_taxon,
                    const int32_t *adj_depth, const double *adj_val, const int32_t *root_depth,
                    const double *tree_weight, int contract_edges, uint64_t seed, int32_t *part,
                    scs_node_stats *stats_out, bool tour_components);

// ---- sharded nodes (shard.cu) -----------------------------------------------------------------------
bool shard_applies(const scs_ctx *ctx, int n);
// A barrier over the ranks on the context's stream (signal every peer, wait for every peer).
int shard_barrier(scs_ctx *ctx);
// Copy [offset, offset + bytes) of this rank's window into the same place of every peer's window.
int shard_push(scs_ctx *ctx, size_t offset, size_t bytes);
// Next epoch / vec buffer for a fused matvec + all-gather (spectral.cu launches the kernel itself).
struct ShardMatvecTicket {
    unsigned long long epoch;
    size_t vec_offset;
    unsigned long long timeout_ns;
};
ShardMatvecTicket shard_next_matvec(scs_ctx *ctx);
int node_split_sharded(scs_ctx *ctx, int n, int T, int64_t L, const int64_t *leaf_offsets, const int32_t *leaf_taxon,
                       const int32_t *adj_depth, const double *adj_val, const int32_t *root_depth,
                       const double *tree_weight, int contract_edges, uint64_t seed, int32_t *part_dev,
                       int32_t *part_host, scs_node_stats *stats);

}  // namespace scs
