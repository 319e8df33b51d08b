// Source trees resident on the device: the forests of one wave of the recursion as flat arrays in HBM, the leaf
// tours derived from them, and their restriction to the children of the wave's nodes -- the device-side
// replacement of the reference's _generate_induced_trees_with_weights
// (/root/reference/src/sc_supertree/scs.py:411-455, PhyloNode.get_sub_tree) and of the host code in forest.cpp.
#pragma once

#include "common.cuh"

struct scs_forest;

namespace scs {

// A grow-only device allocation outside the per-node workspace slots (stream-ordered, like reserve()).
struct GrowBuf {
    void *ptr = nullptr;
    size_t bytes = 0;
    template <typename T>
    T *as() const { return static_cast<T *>(ptr); }
};
int grow(scs_ctx *ctx, GrowBuf &buf, size_t bytes);
void release(scs_ctx *ctx, GrowBuf &buf);

// The trees of every sub-problem ("job") of one wave, concatenated: nodes in depth-first pre-order per tree.
struct DevForest {
    int64_t trees = 0, nodes = 0, leaves = 0;  // host copies of the totals (leaves: tips that appear in tours)
    GrowBuf tree_off, leaf_off;                // int64 [trees + 1]: first node / first tour position of a tree
    GrowBuf parent, size, taxon;               // int32 [nodes]: parent within the tree (-1 root), subtree size, taxon or -1
    GrowBuf length, support;                   // double [nodes], NaN = missing; only kept when the weighting reads them
    GrowBuf weight;                            // double [trees]
    GrowBuf tree_job;                          // int32 [trees]: the job (sub-problem of the wave) the tree belongs to
    bool has_length = false, has_support = false;
    void free_all(scs_ctx *ctx);
};

// Leaf tours of a wave (device): the arrays the graph-build kernels read (absolute leaf offsets = forest.leaf_off).
struct DevTours {
    GrowBuf leaf_taxon, adj_depth, root_depth;  // int32 [leaves], [leaves], [trees]
    GrowBuf adj_val;                            // double [leaves]
    GrowBuf depth_s, val_s;                     // scratch per forest node
    void free_all(scs_ctx *ctx);
};

// What the host learns about the jobs a restriction produced.
struct DevJobInfo {
    int32_t trees;        // source trees kept (>= 2 tips of the job)
    int32_t tree_begin;   // first tree of the job in the new forest
    int64_t leaf_begin;   // first tour position
    int64_t node_begin;   // first forest node
    int64_t first_tree_nodes;  // nodes of its first tree (the single-tree shortcut copies that tree, scs.py:96-98)
    int64_t pair_visits;  // sum over its trees of k (k - 1)
};

// Host forest -> device (job 0 owns every tree).  weighting decides which per-node values travel.
// cooperative (every rank of a connected shard group calls this with the same forest): rank r sends only the r-th
// slice of the per-node arrays over PCIe, into its exchange window, and the ranks gather the other slices from each
// other's windows over NVLink -- the host link carries the forest once per box instead of once per GPU.
int devforest_upload(scs_ctx *ctx, const scs_forest *host, int weighting, DevForest *out, bool cooperative = false);

// Tours of every tree of the forest; taxon_vertex_dev[x] = vertex id of taxon x inside its job.
// Sets *bootstrap_missing_host if a bootstrap weighting met a missing support at an LCA (the reference raises
// TypeError there, scs.py:655-657).  Asynchronous except for that flag, which is read at the next synchronisation
// the caller does: pass a device flag to check later.
int devforest_tours(scs_ctx *ctx, const DevForest &forest, int weighting, const int32_t *taxon_vertex_dev, DevTours *tours,
                    int32_t *flags_dev);

// Restriction of a wave's forest to the children of its jobs.
//   src jobs j = 0..J-1: trees [job_tree_begin[j], job_tree_begin[j + 1]), nodes [job_node_begin[j],
//   job_node_begin[j + 1]); job j was split into job_parts[j] parts (0: not split), numbered globally from
//   job_part_base[j]; owner_dev[x] = global part of taxon x, or -1 (the taxon needs no restricted trees);
//   part_newjob[p] = job of part p in the new forest, or -1.
// A tree is restricted to every part that keeps at least two of its tips (scs.py:447-448), exactly as
// PhyloNode.get_sub_tree(names, ignore_missing=True, as_rooted=True): tips outside the part vanish, unary nodes are
// merged into their child with  length(node) + length(child)  bottom-up, the new root loses its length.
// The new forest is ordered by new job, trees in source order.  info[new_jobs] and present_host[num_taxa] (1 where a
// taxon is still a tip of a kept tree) are filled before the call returns, by its one synchronisation (two when a
// split into many parts makes the bound of the workspace too large and its exact size is read back first).
int devforest_restrict(scs_ctx *ctx, const DevForest &src, int num_jobs, const int32_t *job_tree_begin,
                       const int64_t *job_node_begin, const int32_t *job_parts, const int32_t *job_part_base, int num_parts,
                       const int32_t *part_newjob, int new_jobs, const int32_t *owner_host, int num_taxa, DevForest *dst,
                       DevJobInfo *info, uint8_t *present_host);

// (parent, taxon) of whole trees of the forest, packed one after the other into host arrays: tree i occupies forest
// nodes [first_node[i], first_node[i] + tree_nodes[i]) (DevJobInfo.node_begin / first_tree_nodes).
int devforest_fetch_trees(scs_ctx *ctx, const DevForest &forest, int count, const int64_t *first_node,
                          const int64_t *tree_nodes, int32_t *parent_out, int32_t *taxon_out);

}  // namespace scs
