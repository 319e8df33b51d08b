/* scs_b200.h -- C ABI of libscs_b200.so, the B200 (sm_100a) engine for the hot path of
 * Spectral Cluster Supertree.
 *
 * The reference (rmcar17/SpectralClusterSupertree) has no FFI: the seam this library fills is
 * the four private Python functions its recursion calls once per recursion node
 * (src/sc_supertree/scs.py:110-134).  Each entry point below names the reference function it
 * replaces.  The graph the reference keeps as dicts of name tuples is dense here:
 * vertex id = rank of the taxon name in sorted(all names of the node); W, C are row-major n x n.
 *
 * Conventions
 *   - every function returns an scs_status (0 = OK, negative = error); no C++ exception and no
 *     torch type crosses this boundary;
 *   - "_dev" pointers are device pointers owned by the caller; functions taking them only
 *     enqueue work on the context's CUDA stream and return without synchronising, unless they
 *     write a host result (then they synchronise the stream before returning);
 *   - functions ending in "_host" take host pointers, copy in, compute on the GPU and copy the
 *     result out before returning (the per-recursion-node call a Python/cgo/JNI caller binds);
 *   - a context owns its workspace and is not thread-safe; use one context per thread per GPU.
 *
 * Source trees are passed as leaf tours: the leaves of every tree in depth-first order plus,
 * for each pair of consecutive leaves, the depth and the weighting value of their lowest common
 * ancestor (see spectralclustersupertree_b200/flatten.py).  The weighting strategy is already
 * folded into adj_val, so the kernels are weighting-agnostic:
 *   one -> 1, depth -> depth of the LCA, branch -> root-to-LCA length, bootstrap -> support
 *   (scs.py:555-567).
 */
#ifndef SCS_B200_H
#define SCS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct scs_ctx scs_ctx;

typedef enum {
    SCS_OK = 0,
    SCS_ERR_INVALID = -1,     /* bad argument (null pointer, negative size, ...) */
    SCS_ERR_CUDA = -2,        /* a CUDA runtime call failed; see scs_last_error */
    SCS_ERR_NO_DEVICE = -3,   /* no usable CUDA device */
    SCS_ERR_TOO_SMALL = -4,   /* fewer than 2 vertices handed to the spectral step
                                 (sklearn raises ValueError there, _spectral.py:699) */
    SCS_ERR_NO_CONVERGE = -5, /* eigensolver hit its restart limit */
    SCS_ERR_INPUT = -6,       /* malformed leaf tour (taxon id out of range, ...) */
    SCS_ERR_EMPTY = -7,       /* a recursion node was left without source trees (the reference raises
                                 ValueError "There must be at least one tree ...", scs.py:63-65) */
    SCS_ERR_PEER = -8         /* a device-side wait for a peer GPU ran out of time (sharded nodes) */
} scs_status;

/* What happened at one recursion node (the "near-ties reported" clause of the parity contract). */
typedef struct {
    int32_t n_components;    /* components of the proper cluster graph (adjacency = co-occurred) */
    int32_t contracted_size; /* vertices handed to the spectral step (n if nothing contracted) */
    int32_t spectral_ran;    /* 1 if the node went through the spectral step */
    int32_t solver;          /* 0 none, 1 trivial (m = 2), 2 dense Jacobi (one CTA), 3 Lanczos */
    int32_t matvecs;         /* operator applications in the Lanczos solver */
    int32_t restarts;
    int32_t tie_flag;        /* bit 0: eigengap lambda_3 - lambda_2 < 1e-7; bit 1: a vertex within 1e-9
                                (relative) of the 2-means boundary; bit 2: eigensolver stopped at its
                                restart limit; bit 3: a degree is negative or not finite; bit 4: the
                                1-D 2-means has more than one Lloyd-stable split, i.e. sklearn's
                                k-means outcome depends on its random initialisation */
    int32_t kmeans_stable_splits; /* number of Lloyd-stable splits of the Fiedler coordinate */
    double eig[3];           /* three smallest eigenvalues of L = I - D^-1/2 W D^-1/2 (eig[0] = 0;
                                eig[2] is the solver's estimate, NaN if not available) */
    double residual;         /* || N y - theta y ||_2 of the Fiedler Ritz pair */
    double margin;           /* min_i |u_i - midpoint| / range(u): distance to the 2-means cut */
    double kmeans_runner_up; /* between-cluster score of the best other stable split / the optimum's
                                (0 if the optimum is the only stable split) */
} scs_node_stats;

/* ---- context ---------------------------------------------------------------------------- */
int scs_version(void);
const char *scs_status_string(int status);
/* Text of the last error raised on this context ("" if none). */
const char *scs_last_error(const scs_ctx *ctx);
/* stream: a cudaStream_t to run on, or NULL to let the context create its own. */
int scs_ctx_create(int device, void *stream, scs_ctx **out);
int scs_ctx_destroy(scs_ctx *ctx);
int scs_ctx_synchronize(scs_ctx *ctx);
/* Number of kernels this context has launched since creation (bench.py's gpu_launches). */
int64_t scs_ctx_launch_count(const scs_ctx *ctx);

/* Bytes the *_host entry points copied host->device / device->host since the context was made. */
int scs_ctx_io_bytes(const scs_ctx *ctx, int64_t *h2d, int64_t *d2h);
/* A CUDA-event stopwatch on the context's stream (stop waits for the stream to reach it). */
int scs_ctx_timer_start(scs_ctx *ctx);
int scs_ctx_timer_stop(scs_ctx *ctx, double *ms);
/* Recursion nodes with at most `limit` vertices (default and maximum 64) run components, contraction
 * and the spectral split in one single-CTA launch (dense Jacobi); larger ones take the staged path
 * (union-find, max-merge, Lanczos).  0 sends every node down the staged path. */
int scs_ctx_set_small_node_limit(scs_ctx *ctx, int limit);
/* Recursion nodes above the small-node limit with at most `limit` vertices (default and maximum 4096) are
 * processed by scs_supertree_build as ONE batch per wave of the recursion: every stage of the node path (graph
 * build, components, contraction, Lanczos steps in lock-step, 2-means) is one launch over all of them.
 * 0 sends them down the per-node staged path instead. */
int scs_ctx_set_medium_node_limit(scs_ctx *ctx, int limit);
/* scs_supertree_build on one GPU keeps the source trees resident on the device for the whole recursion: tours and
 * the restriction of the trees to the children of a split (scs.py:411-455) are computed there (on = 1, the default).
 * on = 0 keeps them on the host (flat arrays restricted by the host threads, tours copied to the device per wave). */
int scs_ctx_set_device_forest(scs_ctx *ctx, int on);
/* Graph build: use the 8-byte {tour position, slot} bucket entries that nodes of 65 536 taxa or more need
 * at every size (on = 1; for tests of that path). */
int scs_ctx_set_wide_entries(scs_ctx *ctx, int on);
/* Graph build: W is symmetric bit for bit, so by default the CTA of row a visits only the pairs (a, b > a) and a
 * second kernel mirrors the triangle (W, the bit matrices) and sums the rows.  on = 1 makes every row CTA visit all
 * its pairs, as the row block of a node that is sharded over several GPUs always does (tests, A/B timing). */
int scs_ctx_set_full_rows(scs_ctx *ctx, int on);
/* Host wall clock spent per stage of the staged (> 64 vertices) node path since the last reset:
 * [0] enqueue graph build + components, [1] wait for them, [2] enqueue contraction, [3] spectral step,
 * [4] result copy, [5] Lanczos iterations within [3]. */
int scs_ctx_stage_seconds(scs_ctx *ctx, double *seconds8, int reset);
/* Evict the L2 cache by writing a 256 MB scratch buffer (benchmark hygiene between timed steps). */
int scs_ctx_flush_l2(scs_ctx *ctx);
/* Per-launch CUDA-event timing of the two heavy kernels on matrices of >= 2048 vertices:
 * kind 0 = Laplacian matvec (units = flops), kind 1 = graph-build row kernel (units = ordered leaf
 * pairs visited, known for host-tour calls).  _read sums and clears the records of one kind:
 * launches, total ms, total algorithmic bytes, total units. */
int scs_ctx_profile_enable(scs_ctx *ctx, int on);
int scs_ctx_profile_read(scs_ctx *ctx, int kind, int64_t *launches, double *ms, double *bytes, double *units);

/* Profiling aid: SM cycles the batched small-node kernel spent, summed over its CTAs since the last reset, in
 * [0] the graph build from the tours and [1] components + contraction + eigensolver + 2-means (device-wide
 * counters: meaningful with one context at a time). */
int scs_debug_small_cycles(scs_ctx *ctx, uint64_t *cycles2, int reset);
/* cudaProfilerStart (on = 1) / cudaProfilerStop (on = 0): brackets the step `ncu --profile-from-start off`
 * captures (bench.py --profile-step). */
int scs_profiler_range(int on);

/* ---- proper cluster graph: replaces _proper_cluster_graph_edges + _dfs_pcg_weights
 *      (scs.py:495-583, 586-663) ---------------------------------------------------------- *
 * in : n vertices, T trees, L leaves in total;
 *      leaf_offsets[T+1] (int64), leaf_taxon[L] (vertex id), adj_depth[L], adj_val[L],
 *      root_depth[T] (the adj_depth value that means "LCA is the root"), tree_weight[T].
 * out: W[n*n]  sum over trees, in tree order, of fl(adj_val(LCA) * tree_weight)   (scs.py:655-657)
 *      C[n*n]  number of trees in which the pair is a proper cluster (may be NULL)  (scs.py:658)
 *      occ[n]  number of trees containing the taxon                                 (scs.py:580-581)
 *      adj_bits[n * scs_bit_words(n)]  bit b of word j of row a = C[a][32j+b] > 0   (scs.py:651-652)
 *      max_bits[...]                   ... = C[a][b] > 0 && C[a][b] == max(occ[a], occ[b])
 *                                      (the max-graph of scs.py:302-313; may be NULL)
 *      degree[n] row sums of W (may be NULL)
 * No atomics touch W: each row is accumulated by one CTA in tree input order, so W is
 * reproducible and symmetric bit for bit. */
int scs_bit_words(int n);
int scs_pcg_build_dev(scs_ctx *ctx, int n, int T, int64_t L, const int64_t *leaf_offsets_dev,
                      const int32_t *leaf_taxon_dev, const int32_t *adj_depth_dev,
                      const double *adj_val_dev, const int32_t *root_depth_dev,
                      const double *tree_weight_dev, double *W_dev, int32_t *C_dev,
                      int32_t *occ_dev, uint32_t *adj_bits_dev, uint32_t *max_bits_dev,
                      double *degree_dev);

/* The same for rows [row0, row1) only: W_rows_dev holds (row1 - row0) x n doubles (row a at (a - row0) * n); the bit
 * matrices and degree keep their full size and are written for those rows; occ is complete.  This is the unit of
 * the row-sharded multi-GPU build (every row is its own tree-ordered sum: no reduction over ranks). */
int scs_pcg_build_rows_dev(scs_ctx *ctx, int n, int T, int64_t L, const int64_t *leaf_offsets_dev,
                           const int32_t *leaf_taxon_dev, const int32_t *adj_depth_dev, const double *adj_val_dev,
                           const int32_t *root_depth_dev, const double *tree_weight_dev, int row0, int row1,
                           double *W_rows_dev, int32_t *occ_dev, uint32_t *adj_bits_dev, uint32_t *max_bits_dev,
                           double *degree_dev);

/* ---- connected components: replaces _get_graph_components (scs.py:458-492) ---------------- *
 * label[v] = smallest vertex id of v's component; *n_components_host receives the count. */
int scs_components_dev(scs_ctx *ctx, int n, const uint32_t *bits_dev, int32_t *label_dev,
                       int32_t *n_components_host);

/* ---- contraction: replaces _contract_proper_cluster_graph (scs.py:261-387) ---------------- *
 * group[v] = contracted vertex holding v, numbered by smallest member; *m_host their number;
 * Wc[m*m] (leading dimension m) = max of W over the existing edges between two groups, 0 where
 * there is none; degree_c[m] = row sums of Wc (may be NULL).  Wc_dev must hold n*n doubles. */
int scs_contract_dev(scs_ctx *ctx, int n, const double *W_dev, const uint32_t *adj_bits_dev,
                     const uint32_t *max_bits_dev, int32_t *group_dev, int32_t *m_host,
                     double *Wc_dev, double *degree_c_dev);

/* ---- spectral bipartition: replaces spectral_cluster_graph (scs.py:210-258), i.e.
 *      sklearn SpectralClustering(2, affinity="precomputed") ------------------------------ *
 * W[m*m] symmetric, zero diagonal.  side[m] in {0,1}: 2-means on the Fiedler coordinate of the
 * normalised Laplacian.  degree_dev may be NULL (computed here).  seed picks the start vector. */
int scs_spectral_bipartition_dev(scs_ctx *ctx, int m, const double *W_dev, const double *degree_dev,
                                 uint64_t seed, int32_t *side_dev, scs_node_stats *stats_host);

/* y = D^-1/2 W D^-1/2 x on device vectors: the Laplacian matvec the eigensolver iterates
 * (exposed for the roofline measurement; inv_sqrt_deg = 1/sqrt(degree), 1 where degree is 0). */
int scs_normalized_matvec_dev(scs_ctx *ctx, int m, const double *W_dev,
                              const double *inv_sqrt_deg_dev, const double *x_dev, double *y_dev);

/* ---- one recursion node ------------------------------------------------------------------- *
 * Replaces the block scs.py:110-134: build the graph, find its components; if it is connected,
 * optionally contract it and split it in two.  part[n] receives, per vertex, the component
 * index (0..n_components-1, numbered by smallest member) when the graph is disconnected,
 * otherwise the side (0/1) of the spectral bipartition.
 * _host: host buffers in and out (copies inside the call, returns after the result landed).
 * _dev : tours and part are device pointers; stats are still written on the host. */
int scs_node_split_host(scs_ctx *ctx, int n, int T, int64_t L, const int64_t *leaf_offsets,
                        const int32_t *leaf_taxon, const int32_t *adj_depth, const double *adj_val,
                        const int32_t *root_depth, const double *tree_weight, int contract_edges,
                        uint64_t seed, int32_t *part, scs_node_stats *stats);
int scs_node_split_dev(scs_ctx *ctx, int n, int T, int64_t L, const int64_t *leaf_offsets_dev,
                       const int32_t *leaf_taxon_dev, const int32_t *adj_depth_dev,
                       const double *adj_val_dev, const int32_t *root_depth_dev,
                       const double *tree_weight_dev, int contract_edges, uint64_t seed,
                       int32_t *part_dev, scs_node_stats *stats_host);

/* Device pointers of the node most recently processed by scs_node_split_* (valid until the
 * next call on this context); for parity tests and profiling.  Any out pointer may be NULL.
 * *n / *m are that node's vertex count and contracted vertex count (0 if it never contracted). */
int scs_node_last_buffers(scs_ctx *ctx, int *n, int *m, double **W_dev, uint32_t **adj_bits_dev,
                          uint32_t **max_bits_dev, int32_t **occ_dev, double **degree_dev,
                          double **Wc_dev, int32_t **group_dev);

/* Plain device memory helpers for callers without a CUDA runtime binding of their own
 * (ctypes / cgo / JNI); synchronous with respect to the context's stream. */
int scs_dev_alloc(scs_ctx *ctx, size_t bytes, void **out);
int scs_dev_free(scs_ctx *ctx, void *ptr);
int scs_memcpy_h2d(scs_ctx *ctx, void *dev, const void *host, size_t bytes);
int scs_memcpy_d2h(scs_ctx *ctx, void *host, const void *dev, size_t bytes);

/* ---- source-tree store (host side): replaces the PhyloNode lists the reference's recursion
 *      carries and _generate_induced_trees_with_weights (scs.py:411-455) -------------------- *
 * A forest holds T trees as flat arrays: nodes in depth-first pre-order, node_offsets[T+1];
 * parent[M] = index of the parent within the tree (-1 for the root, always < the node's own
 * index); length[M], support[M] with NaN for "missing" (either array may be NULL = all missing);
 * taxon[M] = global taxon id for tips (0..num_taxa-1), -1 for internal nodes.  Global taxon ids
 * are ranks in the sorted list of all tip names, so increasing id = sorted name order. */
typedef struct scs_forest scs_forest;
/* Host threads the forest operations and the recursion driver may use (process-wide; 0 = the OpenMP
 * default, which launchers such as torchrun pin to 1 through OMP_NUM_THREADS). */
int scs_set_host_threads(int threads);
int scs_forest_create(int T, const int64_t *node_offsets, const int32_t *parent, const double *length,
                      const double *support, const int32_t *taxon, const double *tree_weight,
                      int num_taxa, scs_forest **out);
/* The same without copying the per-node arrays: the forest refers to the caller's parent / length / support / taxon
 * arrays, which must stay alive and unchanged until scs_forest_destroy (node_offsets and tree_weight are copied).
 * For callers that hold the flat trees anyway: at 50 000 taxa x 5 000 trees the copy is a gigabyte per process. */
int scs_forest_create_view(int T, const int64_t *node_offsets, const int32_t *parent, const double *length,
                           const double *support, const int32_t *taxon, const double *tree_weight, int num_taxa,
                           scs_forest **out);
/* Why the last scs_forest_create on this thread returned SCS_ERR_INPUT ("" if it did not): a malformed
 * pre-order tree, or a taxon that labels two tips of one source tree (rejected: the graph kernels give every
 * leaf of a tree its own column). */
const char *scs_forest_last_error(void);
int scs_forest_destroy(scs_forest *f);
/* Newick text (one tree per line, as load_trees reads it: /root/reference/src/sc_supertree/load.py:21-22)
 * straight into a forest, without node objects.  Label rules are those of cogent3.make_tree that the
 * reference's tests rely on: ':x' is a branch length, a numeric label on an internal node is its support
 * (tests/test_spectral_cluster_supertree.py:186-187, 217-219); every tree gets weight 1.  *names receives the
 * sorted tip names (global taxon id = position), each terminated by a NUL byte, *names_bytes their total
 * size; release it with scs_free.  SCS_ERR_INPUT on a syntax error (scs_newick_last_error: "line N: ..."). */
int scs_forest_parse_newick(const char *text, size_t bytes, scs_forest **out, char **names, size_t *names_bytes,
                            int *num_taxa);
const char *scs_newick_last_error(void);
/* The flat supertree (scs_supertree_nodes: parent[i] < i, taxon >= 0 on tips) as Newick text without node objects:
 * replaces PhyloNode.write of the result (/root/reference/src/sc_supertree/cli.py:39).  names: the sorted tip
 * names, NUL-terminated one after the other (as scs_forest_parse_newick returns them).  *text receives a
 * NUL-terminated string ending in ';' (release with scs_free), *text_bytes its length. */
int scs_flat_tree_newick(int64_t num_nodes, const int32_t *parent, const int32_t *taxon, const char *names,
                         size_t names_bytes, int num_taxa, char **text, size_t *text_bytes);
/* scs_flat_tree_newick with a numeric label after every internal non-root node whose value is finite
 * (printf "%.*f", digits, 0 <= digits <= 17); NaN = no label.  value[num_nodes] is indexed like parent. */
int scs_flat_tree_newick_values(int64_t num_nodes, const int32_t *parent, const int32_t *taxon, const char *names,
                                size_t names_bytes, int num_taxa, const double *value, int digits, char **text,
                                size_t *text_bytes);
void scs_free(void *ptr);
int scs_forest_num_trees(const scs_forest *f);
int64_t scs_forest_num_nodes(const scs_forest *f);
int64_t scs_forest_num_leaves(const scs_forest *f);
int scs_forest_num_taxa(const scs_forest *f);
/* sum over trees of k (k - 1): ordered leaf pairs the graph build visits */
int64_t scs_forest_pair_visits(const scs_forest *f);
int scs_forest_tree_info(const scs_forest *f, int t, int64_t *num_nodes, double *weight, int32_t *source);
int scs_forest_tree(const scs_forest *f, int t, int32_t *parent, double *length, double *support,
                    int32_t *taxon);
/* present[num_taxa] = 1 where the taxon is a tip of some tree (scs.py:708-725); returns the
 * number present, or a negative status. */
int scs_forest_taxa(const scs_forest *f, uint8_t *present);
/* Restrict every tree to the taxa with keep[taxon] != 0, as PhyloNode.get_sub_tree(names,
 * ignore_missing=True, as_rooted=True) does; trees left with < 2 tips are dropped with their
 * weight (scs.py:444-453). */
int scs_forest_induce(const scs_forest *f, const uint8_t *keep, scs_forest **out);
/* All the restrictions of one recursion node (the loop scs.py:139-155) in one call, spread over the host
 * threads by (part, tree): out[c] = the forest restricted to the taxa x with part[x] == c, c = 0..count-1
 * (other values of part[x] drop the taxon).  present[num_taxa] (may be NULL) must be zero on entry and is
 * set to 1 for every taxon that is still a tip of some restricted tree. */
int scs_forest_induce_parts(const scs_forest *f, const int32_t *part, int count, scs_forest **out,
                            uint8_t *present);
/* Leaf tours of the forest for one weighting (0 one, 1 branch, 2 depth, 3 bootstrap;
 * scs.py:555-567); local_id[num_taxa] maps global taxon id -> vertex id.  Output arrays are
 * sized by scs_forest_num_trees / scs_forest_num_leaves. */
int scs_forest_tours(const scs_forest *f, int weighting, const int32_t *local_id, int64_t *leaf_offsets,
                     int32_t *leaf_taxon, int32_t *adj_depth, double *adj_val, int32_t *root_depth,
                     double *tree_weight);
/* One recursion node straight from a forest (scs.py:102-134): vertices = taxa present, in
 * increasing global id.  taxa_out / part_out must hold num_taxa entries; *n_out receives n. */
int scs_forest_split(scs_ctx *ctx, const scs_forest *f, int weighting, int contract_edges, uint64_t seed,
                     int32_t *n_out, int32_t *taxa_out, int32_t *part_out, scs_node_stats *stats);

/* ---- many small recursion nodes in one launch --------------------------------------------- *
 * Nodes with at most 64 vertices, one CTA each: graph build, components, contraction and spectral
 * split (scs.py:108-134 for every node of the batch).  The nodes' tours are concatenated:
 * node b owns leaves [leaf_base, leaf_base + its leaf count), trees [tree_base, tree_base + num_trees)
 * of root_depth / tree_weight, offsets leaf_offsets[tree_base + b .. tree_base + b + num_trees]
 * (relative to leaf_base, starting at 0) and vertices [vertex_base, vertex_base + n) of part. */
typedef struct {
    int32_t n;
    int32_t num_trees;
    int64_t leaf_base;
    int64_t tree_base;
    int64_t vertex_base;
} scs_small_node;
int scs_nodes_split_small_host(scs_ctx *ctx, int num_nodes, const scs_small_node *nodes, int64_t L_total,
                               int64_t T_total, const int64_t *leaf_offsets, const int32_t *leaf_taxon,
                               const int32_t *adj_depth, const double *adj_val, const int32_t *root_depth,
                               const double *tree_weight, int contract_edges, int32_t *part,
                               scs_node_stats *stats);

/* Same, on device-resident inputs and outputs; only enqueues the launch (stats_dev is a device array
 * of num_nodes scs_node_stats). */
int scs_nodes_split_small_dev(scs_ctx *ctx, int num_nodes, const scs_small_node *nodes_dev,
                              const int64_t *leaf_offsets_dev, const int32_t *leaf_taxon_dev,
                              const int32_t *adj_depth_dev, const double *adj_val_dev,
                              const int32_t *root_depth_dev, const double *tree_weight_dev,
                              int contract_edges, int32_t *part_dev, scs_node_stats *stats_dev);

/* ---- a batch of medium-sized recursion nodes, one launch per stage ------------------------------------ *
 * Nodes of at most 4096 vertices (scs_supertree_build sends those above the small-node limit): the block
 * scs.py:108-134 for every node of the batch, every stage -- graph build, components, contraction, the Lanczos
 * steps in lock-step, 2-means -- ONE launch over all of them.  Host arrays: node_n[num_nodes],
 * tree_begin[num_nodes + 1] (node b owns trees [tree_begin[b], tree_begin[b + 1]) of the concatenated tours),
 * part_offset[num_nodes] (where its labels go in part_dev), seeds[num_nodes].  Device arrays: the tours of all
 * nodes, concatenated, leaf_offsets[T + 1] ABSOLUTE; leaf_taxon holds vertex ids local to the node.
 * stats[num_nodes] and needs_rerun[num_nodes] are host arrays; needs_rerun[b] = 1 asks the caller to send node b
 * through scs_node_split_* instead (eigensolver restart after 256 steps, or the deflated second run that settles a
 * repeated Fiedler eigenvalue: rare).  Returns after the results landed. */
int scs_nodes_split_medium_dev(scs_ctx *ctx, int num_nodes, const int32_t *node_n, const int32_t *tree_begin,
                               const int64_t *part_offset, const uint64_t *seeds, int T, int64_t L,
                               const int64_t *leaf_offsets_dev, const int32_t *leaf_taxon_dev, const int32_t *adj_depth_dev,
                               const double *adj_val_dev, const int32_t *root_depth_dev, const double *tree_weight_dev,
                               int contract_edges, int32_t *part_dev, scs_node_stats *stats, uint8_t *needs_rerun);

/* ---- the whole recursion (scs.py:96-174) as a native work-list ------------------------------- *
 * Breadth-first over the independent sub-problems, wave by wave, with the source trees resident on the
 * device (uploaded once; leaf tours and the restriction to the children of every split, scs.py:411-455, are
 * computed there): the frontier nodes up to the small-node limit (scs_ctx_set_small_node_limit, default 32
 * taxa) are split in ONE launch, those up to 4096 taxa go through every stage together as one batch, larger
 * ones one by one (row-sharded over the GPUs of a connected shard group).  The result is the supertree
 * as flat arrays: parent[i] < i (-1 for the root), taxon[i] = global taxon id for tips, -1 for
 * internal nodes; children are in index order.  With record_nodes != 0 every recursion node that
 * reached the GPU is kept (vertices, part, stats) for node-by-node parity checks. */
typedef struct scs_supertree scs_supertree;
int scs_supertree_build(scs_ctx *ctx, const scs_forest *forest, int weighting, int contract_edges,
                        uint64_t seed, int record_nodes, scs_supertree **out);
/* One job over `world` GPUs, one process each, no collective on the data path: every rank runs the
 * first waves redundantly (deterministic kernels => identical frontier and identical output prefix),
 * then the frontier is dealt out by estimated cost and each rank finishes its own sub-problems.
 * Output nodes [0, scs_supertree_shared_prefix) are the same on every rank; the caller appends the
 * other ranks' nodes past the prefix (parents >= prefix shift by the append offset). */
int scs_supertree_build_sharded(scs_ctx *ctx, const scs_forest *forest, int weighting, int contract_edges,
                                uint64_t seed, int record_nodes, int rank, int world, scs_supertree **out);
/* The source trees uploaded once and kept in HBM between builds: scs_supertree_build does
 * scs_device_forest_create + scs_supertree_build_resident + scs_device_forest_destroy; a caller that builds several
 * supertrees from the same trees (other weights of the spectral step, a benchmark with inputs resident in HBM) keeps
 * the device forest.  The weighting decides which per-node values are uploaded (branch: lengths, bootstrap:
 * supports).  With world > 1 the build is the cooperative one (exchange windows must be connected). */
typedef struct scs_device_forest scs_device_forest;
int scs_device_forest_create(scs_ctx *ctx, const scs_forest *forest, int weighting, scs_device_forest **out);
int scs_device_forest_destroy(scs_device_forest *forest);
int64_t scs_device_forest_bytes(const scs_device_forest *forest);
int scs_supertree_build_resident(scs_ctx *ctx, const scs_device_forest *forest, int contract_edges, uint64_t seed,
                                 int record_nodes, int rank, int world, scs_supertree **out);
int64_t scs_supertree_shared_prefix(const scs_supertree *tree);
/* Recursion nodes (records [0, this)) processed before the frontier was dealt out: the same on every
 * rank, and the ones that are shared out over the GPUs when a shard group is connected. */
int64_t scs_supertree_shared_records(const scs_supertree *tree);
/* Per wave of the breadth-first recursion: number of sub-problems and the largest one's taxon count.
 * Returns the number of waves; either array may be NULL (size them with scs_supertree_counters). */
int scs_supertree_wave_info(const scs_supertree *tree, int32_t *tasks, int32_t *max_n);
/* Per wave, 3 doubles: seconds in GPU splits, in forest restriction, in the whole wave. */
int scs_supertree_wave_seconds(const scs_supertree *tree, double *seconds3);
int scs_supertree_destroy(scs_supertree *tree);
int64_t scs_supertree_num_nodes(const scs_supertree *tree);
int scs_supertree_nodes(const scs_supertree *tree, int32_t *parent, int32_t *taxon);
int scs_supertree_counters(const scs_supertree *tree, int64_t *nodes_small, int64_t *nodes_large,
                           int64_t *waves, int64_t *pair_visits);
/* Host wall-clock seconds the build spent in: [0] large-node splits, [1] small-node batches,
 * [2] restricting forests, [3] flattening tours. */
int scs_supertree_seconds(const scs_supertree *tree, double *seconds4);
/* Recursion nodes that went through the batched medium-node path, how many of those had to be re-run through the
 * per-node path (eigensolver restart / repeated-eigenvalue check), and the host seconds spent in the batches. */
int scs_supertree_medium_info(const scs_supertree *tree, int64_t *nodes_medium, int64_t *nodes_rerun, double *seconds);
int64_t scs_supertree_num_records(const scs_supertree *tree);
int scs_supertree_record_size(const scs_supertree *tree, int64_t index);
/* Wave of the breadth-first recursion (0 = the top-level node) in which record `index` was processed. */
int scs_supertree_record_wave(const scs_supertree *tree, int64_t index);
int scs_supertree_record(const scs_supertree *tree, int64_t index, int32_t *taxa, int32_t *part,
                         scs_node_stats *stats);

/* ---- source-tree support of the clades of a supertree ----------------------------------------------------- *
 * Source-tree support of every clade of a supertree (parent[i] < i, taxon >= 0 on tips, ids in the forest's id
 * space, no repeated taxon).  For internal node u and source tree t, A = leaves(u) restricted to the taxa X_t that t
 * shares with the supertree is classified against t restricted to X_t (as scs_forest_induce restricts): irrelevant
 * (|A| < 2 or A = X_t), support (A is one of its clusters), conflict (A overlaps one of its non-trivial clusters
 * without nesting), permitted (otherwise).  counts[3 * num_nodes]: support, conflict, permitted per node (tips: 0);
 * weighted (may be NULL) the same summed with the tree weights, in tree order; per_tree[4 * T]: shared clusters,
 * source clusters, supertree clusters and their rooted Robinson-Foulds distance, all over the non-trivial clusters on
 * X_t (0 when |X_t| < 2).  SCS_ERR_INPUT for a malformed supertree.  Returns after the results landed. */
int scs_supertree_support(scs_ctx *ctx, const scs_forest *sources, int64_t num_nodes, const int32_t *parent,
                          const int32_t *taxon, int32_t *counts, double *weighted, int32_t *per_tree);

/* Rooted triplet fit of the same supertree (validated as in scs_supertree_support; SCS_ERR_INPUT if malformed)
 * against every source tree t, both restricted to the k taxa X_t they share.  A triplet {a, b, c} of X_t is resolved
 * as ab|c when LCA(a, b) lies strictly below LCA(a, b, c), a fan otherwise.  per_tree[5 * T], int64 per tree: k,
 * triplets resolved in the restricted source tree, triplets resolved in the restricted supertree, triplets resolved
 * the same way in both (agree) and resolved differently (contradict); all but k are 0 when k < 3.  SCS_ERR_INVALID if
 * a leaf of the supertree lies deeper than its shared-memory Fenwick tree allows (about 29 000 levels).  Returns
 * after the results landed. */
int scs_supertree_triplets(scs_ctx *ctx, const scs_forest *sources, int64_t num_nodes, const int32_t *parent,
                           const int32_t *taxon, int64_t *per_tree);

/* The same triplets credited to their taxa (validated and failing as scs_supertree_triplets).  For every taxon p,
 * summed over the source trees t with p in X_t and k = |X_t| >= 3, int64 per_taxon[6 * num_taxa], row p: the number
 * of such trees, the triplets of X_t that contain p (sum of C(k - 1, 2)), and those of them resolved in the restricted
 * source tree, resolved in the restricted supertree, resolved the same way in both (agree) and resolved differently
 * (contradict).  Rows are indexed by the forest's taxon id; taxa that are not tips of the supertree are all zero, and
 * a tree of one tip adds nothing.  weighted (may be NULL) [3 * num_taxa], row p: resolved source, agree and
 * contradict summed over the same trees in tree order as acc = acc + w_t * count, without fused multiply-add.
 * SCS_ERR_INVALID if a leaf of the supertree lies deeper than the three shared-memory arrays of a row allow (about
 * 19 000 levels).  Returns after the results landed. */
int scs_supertree_taxon_triplets(scs_ctx *ctx, const scs_forest *sources, int64_t num_nodes, const int32_t *parent,
                                 const int32_t *taxon, int64_t *per_taxon, double *weighted);

/* MRP (matrix representation with parsimony) score of the same supertree (validated as in scs_supertree_support;
 * SCS_ERR_INPUT if malformed).  Every non-trivial cluster c (2 <= |c| < k) of source tree t restricted to the k taxa
 * X_t it shares with the supertree is one binary character: 1 on c, 0 on X_t \ c, missing on the other tips.  Its
 * length is the minimum number of state changes on the supertree (Fitch/Hartigan; polytomies are hard, unary nodes
 * pass their child's set up) with an all-0 outgroup above the root.  per_tree[4 * T], int64 per tree: k, characters,
 * their summed length (steps) and the characters of length 1 (exactly the clusters of the restricted supertree); all
 * but k are 0 when k < 3.  SCS_ERR_INVALID if a leaf of the supertree lies deeper than the shared-memory stack of a
 * character allows (about 29 000 levels, as scs_supertree_triplets), or if the supertree has more tips than the
 * shared-memory bitmap of a tree allows (about 925 000, as scs_supertree_support).  Returns after the results
 * landed. */
int scs_supertree_mrp(scs_ctx *ctx, const scs_forest *sources, int64_t num_nodes, const int32_t *parent,
                      const int32_t *taxon, int64_t *per_tree);

/* Rooted Robinson-Foulds distances between every pair of source trees of the forest, each pair restricted to the k
 * taxa X it shares (as scs_forest_induce restricts; no supertree is involved).  Three caller-owned T x T row-major
 * int32 arrays: shared_taxa[i][j] = k (symmetric; the diagonal is the tree's tip count); clusters[i][j] = the
 * non-trivial clusters (2 <= |c| < k) of tree i restricted to X (not symmetric: row i counts tree i's clusters); common
 * = the clusters the two restrictions have in common (symmetric).  clusters and common are 0 where k < 3.  The rooted
 * RF distance is clusters[i][j] + clusters[j][i] - 2 common[i][j]; with tree i as the supertree, scs_supertree_support
 * gives for source tree j: shared clusters = common[i][j], source clusters = clusters[j][i], supertree clusters =
 * clusters[i][j].  Tree weights do not enter.  SCS_ERR_INVALID if the forest has more taxa than the shared-memory
 * bitmap of a pair allows (about 925 000) or more trees than the grid of 64 x 64 pair tiles allows (about 4 million).
 * Returns after the results landed. */
int scs_forest_pairwise_rf(scs_ctx *ctx, const scs_forest *forest, int32_t *shared_taxa, int32_t *clusters,
                           int32_t *common);

/* ---- one recursion node over several GPUs of one NVLink box (one process per GPU) ------------- *
 * The reference is single-process (scs.py:239 n_jobs=1); this is the B200 answer to its largest
 * recursion nodes.  A node with >= min_n taxa is ROW-SHARDED: rank r builds and keeps rows
 * [r * ceil(n / world), ...) of W (every row is its own tree-ordered sum, so the result stays bit-exact),
 * pushes its adjacency-bit rows and degrees into the peers' exchange windows over NVLink, and every
 * Lanczos step is one kernel that computes the rank's slice of y = D^-1/2 W D^-1/2 x, stores it into
 * every peer's window and waits for the peers' slices (compute + all-gather + barrier in one launch).
 * Components, contraction groups and the Lanczos vector work are replicated, so every rank ends with
 * the same partition as the single-GPU path, bit for bit.
 *
 * Protocol: every rank calls scs_shard_create (allocates its window, returns a cudaIpcMemHandle_t as
 * 64 opaque bytes), the caller all-gathers the handles (torch.distributed, MPI, a file ...), every
 * rank calls scs_shard_connect_ipc with all of them in rank order.  While engaged, every rank must
 * issue the same sequence of node calls (scs_node_split_* / scs_supertree_build_sharded do).
 * scs_shard_destroy must only be called after all ranks finished their last node (host barrier). */
#define SCS_IPC_HANDLE_BYTES 64
int scs_shard_create(scs_ctx *ctx, int rank, int world, int n_max, unsigned char *handle_out);
int scs_shard_connect_ipc(scs_ctx *ctx, const unsigned char *handles /* world * 64 bytes */);
/* Peers that live in the same process (one context per GPU, or several on one GPU): plain pointers. */
int scs_shard_window(scs_ctx *ctx, void **window_dev, size_t *bytes);
int scs_shard_connect_ptrs(scs_ctx *ctx, void *const *windows /* world pointers, own included */);
/* While engaged, nodes with min_n <= n <= n_max handed to this context take the sharded path. */
int scs_shard_engage(scs_ctx *ctx, int on);
/* min_n: smallest node that is shared out (default 4096; <= 0 keeps it); timeout_seconds: bound on
 * every device-side wait for a peer (default 20; <= 0 keeps it). */
int scs_shard_configure(scs_ctx *ctx, int min_n, double timeout_seconds);
/* A barrier over the ranks through the windows (signal every peer, wait for every peer). */
int scs_shard_barrier(scs_ctx *ctx);
/* Recursion nodes this context processed on the sharded path. */
int64_t scs_shard_nodes(const scs_ctx *ctx);
int scs_shard_destroy(scs_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* SCS_B200_H */
