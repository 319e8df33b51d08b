// The supertree recursion with the source trees resident on the device.
//
// Same control flow as driver.cu (the reference's construct_supertree, /root/reference/src/sc_supertree/scs.py:96-174,
// breadth-first over the independent sub-problems), but the forests never come back to the host: the original trees
// are uploaded once; per wave the leaf tours of every sub-problem are derived on the device (devforest.cu: df_tours),
// the nodes are split there (small batch / medium batch / per-node path, all reading the same device-resident
// tours), and the trees are restricted to the children on the device (devforest_restrict, the replacement of
// _generate_induced_trees_with_weights, scs.py:411-455).  What crosses the bus per wave is bookkeeping: vertex ids
// and part owners of the taxa down (4 bytes per taxon each), partitions, per-node records, per-child tree counts and
// a presence byte per taxon up.  The host keeps what the reference keeps outside its tree objects: which taxa belong
// to which sub-problem, and the output tree.

#include "common.cuh"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <thread>

#include "devforest.cuh"
#include "driver.hpp"
#include "forest.hpp"

// Source trees uploaded once and kept on the device between builds (scs_device_forest_create): the arrays plus what the
// recursion needs to know about them on the host.
struct scs_device_forest {
    scs::DevForest trees;
    int weighting = 0;
    int num_taxa = 0;
    std::vector<int32_t> taxa;  // taxa present, ascending
    int64_t first_tree_nodes = 0, pair_visits = 0, leaves = 0;
    scs_ctx *owner = nullptr;
};

namespace scs {

namespace {

struct Stopwatch {
    double *sink;
    std::chrono::steady_clock::time_point t0;
    explicit Stopwatch(double *s) : sink(s), t0(std::chrono::steady_clock::now()) {}
    ~Stopwatch() { *sink += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count(); }
};

// A sub-problem of the current wave: a set of taxa and its trees in the wave's device forest.
struct Job {
    int32_t slot = 0;           // output node it fills in
    std::vector<int32_t> taxa;  // taxa present in its trees, ascending (vertex id = rank; scs.py:708-725)
    DevJobInfo where{};         // its trees / leaves / nodes in the wave's forest
    int64_t leaves = 0;         // tour positions of its trees
    bool shared = false;        // cooperative build: every rank holds and processes this job (row-sharded over the GPUs)
};

__global__ void relative_offsets(int count, const int64_t *__restrict__ absolute, int64_t *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) out[i] = absolute[i] - absolute[0];
}

// What a context keeps between builds: the two alternating wave forests, the tours, the small per-wave arrays and the
// device copy of the source trees of scs_supertree_build (grow-only: after the first build of a size nothing is
// allocated any more).
struct DriverCache {
    DevForest forest[2];
    DevTours tours;
    GrowBuf vertex_dev, offsets_rel, part_dev, flags_dev;
    scs_device_forest resident;
};

void release_driver_cache(scs_ctx *ctx, void *raw) {
    DriverCache *cache = static_cast<DriverCache *>(raw);
    cache->forest[0].free_all(ctx);
    cache->forest[1].free_all(ctx);
    cache->tours.free_all(ctx);
    for (GrowBuf *b : {&cache->vertex_dev, &cache->offsets_rel, &cache->part_dev, &cache->flags_dev}) release(ctx, *b);
    cache->resident.trees.free_all(ctx);
    cudaStreamSynchronize(ctx->stream);
    delete cache;
}

DriverCache &driver_cache(scs_ctx *ctx) {
    if (!ctx->driver_cache) {
        ctx->driver_cache = new DriverCache();
        ctx->driver_cache_release = release_driver_cache;
    }
    return *static_cast<DriverCache *>(ctx->driver_cache);
}

class DeviceDriver {
  public:
    DeviceDriver(scs_ctx *ctx, int weighting, int contract_edges, uint64_t seed, bool record, int rank, int world,
                 scs_supertree *out)
        : ctx_(ctx), weighting_(weighting), contract_(contract_edges), seed_(seed), record_(record), rank_(rank),
          world_(world), out_(*out), cache_(driver_cache(ctx)), forest_(cache_.forest), tours_(cache_.tours),
          vertex_dev_(cache_.vertex_dev), offsets_rel_(cache_.offsets_rel), part_dev_(cache_.part_dev),
          flags_dev_(cache_.flags_dev) {}

    ~DeviceDriver() {
        if (tours_ready_) cudaEventDestroy(tours_ready_);
        cudaStreamSynchronize(ctx_->stream);
    }

    int run(const scs_device_forest *root) {
        num_taxa_ = root->num_taxa;
        root_ = &root->trees;
        int rc;
        vertex_.assign(static_cast<size_t>(num_taxa_ > 0 ? num_taxa_ : 1), -1);
        owner_.assign(vertex_.size(), -1);
        present_.assign(vertex_.size(), 0);
        if ((rc = grow(ctx_, flags_dev_, 64 * sizeof(int32_t)))) return rc;
        SCS_CUDA(ctx_, cudaMemsetAsync(flags_dev_.ptr, 0, 64 * sizeof(int32_t), ctx_->stream));

        const ShardState &sh = ctx_->shard;
        cooperative_ = world_ > 1 && sh.connected && sh.world == world_ && sh.rank == rank_;
        std::vector<Job> wave(1), next;
        wave[0].slot = add(-1, -1, cooperative_);
        wave[0].taxa = root->taxa;
        wave[0].where.trees = static_cast<int32_t>(root->trees.trees);
        wave[0].where.first_tree_nodes = root->first_tree_nodes;
        wave[0].where.pair_visits = root->pair_visits;
        wave[0].leaves = root->leaves;
        cur_ = -1;  // the first wave reads the resident forest; its children go to forest_[0]
        if (cooperative_) {
            load_.assign(static_cast<size_t>(world_), 0.0);
            const int n_root = static_cast<int>(wave[0].taxa.size());
            wave[0].shared = stays_shared(n_root);
            if (!wave[0].shared && deal(n_root) != rank_) wave.clear();  // a small job: one rank does it all
        }
        while (!wave.empty()) {
            out_.waves += 1;
            int32_t max_n = 0;
            for (const Job &job : wave) max_n = std::max<int32_t>(max_n, static_cast<int32_t>(job.taxa.size()));
            out_.wave_tasks.push_back(static_cast<int32_t>(wave.size()));
            out_.wave_max_n.push_back(max_n);
            const double before_gpu = out_.seconds[0] + out_.seconds[1] + out_.medium_seconds, before_restrict = out_.seconds[2];
            const double before[6] = {out_.seconds[0], out_.seconds[1], out_.medium_seconds, out_.seconds[3], out_.seconds[2],
                                      restrict_device_s_};
            const auto wave_start = std::chrono::steady_clock::now();
            next.clear();
            if ((rc = process_wave(wave, next))) return rc;
            out_.wave_seconds.push_back(out_.seconds[0] + out_.seconds[1] + out_.medium_seconds - before_gpu);
            out_.wave_seconds.push_back(out_.seconds[2] - before_restrict);
            out_.wave_seconds.push_back(std::chrono::duration<double>(std::chrono::steady_clock::now() - wave_start).count());
            if (trace_)
                std::fprintf(stderr,
                             "[scs devdriver] wave %2d: tasks %5zu max_n %6d | large %7.3f small %7.3f medium %7.3f tours %6.3f "
                             "children %6.3f (device restriction %6.3f) | wave %7.3f ms\n",
                             static_cast<int>(out_.waves - 1), wave.size(), max_n, 1e3 * (out_.seconds[0] - before[0]),
                             1e3 * (out_.seconds[1] - before[1]), 1e3 * (out_.medium_seconds - before[2]),
                             1e3 * (out_.seconds[3] - before[3]), 1e3 * (out_.seconds[2] - before[4]),
                             1e3 * (restrict_device_s_ - before[5]), 1e3 * out_.wave_seconds.back());
            wave.swap(next);
        }
        ctx_->shard.engaged = false;
        if (cooperative_) finish_cooperative();
        return SCS_OK;
    }

  private:
    bool stays_shared(int size) const { return cooperative_ && size >= ctx_->shard.min_n; }
    int deal(int size) {
        const double n = static_cast<double>(size);
        const int r = static_cast<int>(std::min_element(load_.begin(), load_.end()) - load_.begin());
        load_[r] += n + n * n / 2.0e5;  // small nodes cost per node (latency), large ones per leaf pair
        return r;
    }
    void finish_cooperative() {
        const int32_t S = static_cast<int32_t>(sh_parent_.size());
        auto final_index = [S](int32_t id) { return id >= 0 ? S + id : (id == -1 ? -1 : -2 - id); };
        std::vector<int32_t> parent(sh_parent_.size() + out_.parent.size()), taxon(parent.size());
        for (int32_t i = 0; i < S; ++i) {
            parent[i] = final_index(sh_parent_[i]);
            taxon[i] = sh_taxon_[i];
        }
        for (size_t j = 0; j < out_.parent.size(); ++j) {
            parent[S + j] = final_index(out_.parent[j]);
            taxon[S + j] = out_.taxon[j];
        }
        out_.parent.swap(parent);
        out_.taxon.swap(taxon);
        out_.shared_prefix = S;
        out_.shared_records = static_cast<int64_t>(sh_records_.size());
        sh_records_.insert(sh_records_.end(), std::make_move_iterator(out_.records.begin()),
                           std::make_move_iterator(out_.records.end()));
        out_.records.swap(sh_records_);
    }

    // ---- output nodes (scs.py:390-408, 728-746) -----------------------------------------------------------------------
    // Node ids: id >= 0 is a node of this rank's own list; id <= -2 is node -2 - id of the shared list (cooperative
    // builds only); -1 is "no parent".
    int32_t add(int32_t parent, int32_t taxon, bool shared) {
        if (shared) {
            sh_parent_.push_back(parent);
            sh_taxon_.push_back(taxon);
            return -2 - static_cast<int32_t>(sh_parent_.size() - 1);
        }
        out_.parent.push_back(parent);
        out_.taxon.push_back(taxon);
        return static_cast<int32_t>(out_.parent.size() - 1);
    }
    void set_taxon(int32_t id, int32_t taxon) {
        if (id >= 0) out_.taxon[id] = taxon;
        else sh_taxon_[-2 - id] = taxon;
    }
    void fill_star(int32_t slot, const int32_t *taxa, int count, bool shared) {  // one name stays a tip, more a star
        if (count == 1) {
            set_taxon(slot, taxa[0]);
            return;
        }
        for (int i = 0; i < count; ++i) add(slot, taxa[i], shared);
    }

    struct Split {
        size_t job = 0;
        int64_t part_at = 0;  // where its labels are in part_
        scs_node_stats stats{};
        int32_t parts = 0, part_base = 0;
    };

    const DevForest &current() const { return cur_ < 0 ? *root_ : forest_[cur_]; }
    DevForest &other() { return forest_[cur_ < 0 ? 0 : 1 - cur_]; }

    int process_wave(std::vector<Job> &wave, std::vector<Job> &next) {
        const DevForest &forest = current();
        int rc;
        // ---- what each sub-problem is (scs.py:96-106) -------------------------------------------------------------------
        std::vector<size_t> single, small, medium, large;
        for (size_t i = 0; i < wave.size(); ++i) {
            const Job &job = wave[i];
            const int n = static_cast<int>(job.taxa.size());
            if (job.where.trees == 0) return fail(ctx_, SCS_ERR_EMPTY, "a component is covered by no source tree (scs.py:63-65)");
            if (job.where.trees == 1) single.push_back(i);
            else if (n <= 2) fill_star(job.slot, job.taxa.data(), n, job.shared);
            else if (job.shared) large.push_back(i);  // row-sharded over the GPUs, every rank in the same order
            else if (n <= ctx_->small_limit && job.where.trees <= kSmallMaxTrees) small.push_back(i);
            else if (n <= ctx_->medium_limit) medium.push_back(i);
            else large.push_back(i);
        }
        if (!single.empty() && (rc = copy_single_trees(wave, single))) return rc;
        std::vector<Split> splits;
        if (!small.empty() || !medium.empty() || !large.empty()) {
            // ---- tours of the whole wave on the device -----------------------------------------------------------------
            {
                Stopwatch sw(&out_.seconds[3]);
                for (const std::vector<size_t> *kind : {&small, &medium, &large})
                    for (size_t i : *kind) {
                        const std::vector<int32_t> &taxa = wave[i].taxa;
                        for (size_t v = 0; v < taxa.size(); ++v) vertex_[taxa[v]] = static_cast<int32_t>(v);
                    }
                if ((rc = upload_ints(vertex_dev_, vertex_.data(), vertex_.size()))) return rc;
                if ((rc = devforest_tours(ctx_, forest, weighting_, vertex_dev_.as<int32_t>(), &tours_, flags_dev_.as<int32_t>())))
                    return rc;
            }
            // ---- split the nodes: labels of all of them land in one array ----------------------------------------------
            int64_t labels = 0;
            for (const std::vector<size_t> *kind : {&large, &medium, &small})
                for (size_t i : *kind) {
                    Split s;
                    s.job = i;
                    s.part_at = labels;
                    labels += static_cast<int64_t>(wave[i].taxa.size());
                    splits.push_back(s);
                    out_.pair_visits += wave[i].where.pair_visits;
                }
            part_.resize(static_cast<size_t>(labels) + 1);
            if ((rc = grow(ctx_, part_dev_, (static_cast<size_t>(labels) + 1) * sizeof(int32_t)))) return rc;
            // The three kinds of nodes run next to each other: the batch of small nodes and the batch of medium nodes
            // each on its own context (stream, workspace) and host thread, the large nodes on this one.  All read the
            // wave's tours and write disjoint ranges of the label array; the other streams wait for the tours.
            const size_t at_medium = large.size(), at_small = large.size() + medium.size();
            // this thread takes the large nodes, else the medium batch, else the small batch; the others go aside
            scs_ctx *small_ctx = ctx_, *medium_ctx = ctx_;
            if (scs_host_threads() >= 2 && ensure_workers(ctx_, 3) == SCS_OK) {
                if (!small.empty() && (!large.empty() || !medium.empty())) small_ctx = ctx_->workers[0];
                if (!medium.empty() && !large.empty()) medium_ctx = ctx_->workers[1];
            }
            if (small_ctx != ctx_ || medium_ctx != ctx_) {
                if (!tours_ready_) SCS_CUDA(ctx_, cudaEventCreateWithFlags(&tours_ready_, cudaEventDisableTiming));
                SCS_CUDA(ctx_, cudaEventRecord(tours_ready_, ctx_->stream));
            }
            int small_rc = SCS_OK, medium_rc = SCS_OK;
            double small_s = 0.0, medium_s = 0.0;
            std::vector<size_t> reruns;
            auto run_small = [&](scs_ctx *ctx) {
                Stopwatch sw(&small_s);
                small_rc = split_small(ctx, wave, small, splits.data() + at_small);
            };
            auto run_medium = [&](scs_ctx *ctx) {
                Stopwatch sw(&medium_s);
                medium_rc = split_medium(ctx, wave, medium, splits.data() + at_medium, reruns);
            };
            auto aside = [&](scs_ctx *ctx, auto &work, int *status) {
                return std::thread([this, ctx, &work, status] {
                    cudaError_t err = cudaSetDevice(ctx_->device);
                    if (err == cudaSuccess) err = cudaStreamWaitEvent(ctx->stream, tours_ready_, 0);
                    if (err != cudaSuccess) {
                        *status = fail(ctx, SCS_ERR_CUDA, "starting a batch next to the other nodes of the wave", err);
                        return;
                    }
                    work(ctx);
                });
            };
            std::thread small_thread, medium_thread;
            if (!small.empty() && small_ctx != ctx_) small_thread = aside(small_ctx, run_small, &small_rc);
            if (!medium.empty() && medium_ctx != ctx_) medium_thread = aside(medium_ctx, run_medium, &medium_rc);
            if (!large.empty()) {
                Stopwatch sw(&out_.seconds[0]);
                for (size_t k = 0; k < large.size() && rc == SCS_OK; ++k) rc = split_large(wave[large[k]], splits[k]);
                out_.nodes_large += static_cast<int64_t>(large.size());
            }
            if (rc == SCS_OK && !medium.empty() && medium_ctx == ctx_) run_medium(ctx_);
            if (rc == SCS_OK && !small.empty() && small_ctx == ctx_) run_small(ctx_);
            if (small_thread.joinable()) small_thread.join();
            if (medium_thread.joinable()) medium_thread.join();
            for (scs_ctx *other : {small_ctx, medium_ctx})
                if (other != ctx_) {
                    if (rc == SCS_OK && (other == small_ctx ? small_rc : medium_rc) != SCS_OK) ctx_->last_error = other->last_error;
                    ctx_->launches += other->launches;
                    ctx_->h2d_bytes += other->h2d_bytes;
                    ctx_->d2h_bytes += other->d2h_bytes;
                    other->launches = other->h2d_bytes = other->d2h_bytes = 0;
                }
            out_.seconds[1] += small_s;
            out_.medium_seconds += medium_s;
            if (rc == SCS_OK) rc = small_rc ? small_rc : medium_rc;
            if (rc) return rc;
            out_.nodes_small += static_cast<int64_t>(small.size());
            out_.nodes_medium += static_cast<int64_t>(medium.size());
            // eigensolver restart / repeated-eigenvalue check of a medium node: the per-node path has both
            for (size_t b : reruns) {
                out_.nodes_rerun += 1;
                if ((rc = split_large(wave[medium[b]], splits[at_medium + b]))) return rc;
            }
            // labels of every node of the wave, and the malformed-input flags, in one copy each
            SCS_CUDA(ctx_, cudaMemcpyAsync(part_.data(), part_dev_.as<int32_t>(), sizeof(int32_t) * static_cast<size_t>(labels),
                                           cudaMemcpyDeviceToHost, ctx_->stream));
            int32_t flags[4] = {0, 0, 0, 0};
            SCS_CUDA(ctx_, cudaMemcpyAsync(flags, flags_dev_.ptr, sizeof(flags), cudaMemcpyDeviceToHost, ctx_->stream));
            SCS_CUDA(ctx_, cudaStreamSynchronize(ctx_->stream));
            ctx_->d2h_bytes += static_cast<int64_t>(sizeof(int32_t)) * labels;
            if (flags[0]) return fail(ctx_, SCS_ERR_INPUT, "leaf tour: taxon id out of range");
            if (flags[1]) return fail(ctx_, SCS_ERR_INPUT, "bootstrap weighting: an internal node without support");
            for (const Split &s : splits)
                if (s.stats.solver == -1) return fail(ctx_, SCS_ERR_TOO_SMALL, "spectral step on a graph contracted to one vertex");
        }
        if (splits.empty()) return SCS_OK;
        // ---- children (scs.py:136-171) ---------------------------------------------------------------------------------
        Stopwatch sw(&out_.seconds[2]);
        return plan_children(wave, splits, next);
    }

    int upload_ints(GrowBuf &dev, const int32_t *host, size_t count) {
        int rc;
        if ((rc = grow(ctx_, dev, count * sizeof(int32_t)))) return rc;
        void *pin_v;
        if ((rc = reserve_pinned(ctx_, count * sizeof(int32_t) + 256, &pin_v))) return rc;
        std::memcpy(pin_v, host, count * sizeof(int32_t));
        SCS_CUDA(ctx_, cudaMemcpyAsync(dev.ptr, pin_v, count * sizeof(int32_t), cudaMemcpyHostToDevice, ctx_->stream));
        // the pinned block is reused by the calls that follow: the copy must have left it
        SCS_CUDA(ctx_, cudaStreamSynchronize(ctx_->stream));
        ctx_->h2d_bytes += static_cast<int64_t>(count * sizeof(int32_t));
        return SCS_OK;
    }

    // topology-only copies of the single remaining trees (scs.py:96-98), fetched in one piece
    int copy_single_trees(const std::vector<Job> &wave, const std::vector<size_t> &single) {
        const int count = static_cast<int>(single.size());
        std::vector<int64_t> first(count), nodes(count);
        int64_t total = 0;
        for (int i = 0; i < count; ++i) {
            first[i] = wave[single[i]].where.node_begin;
            nodes[i] = wave[single[i]].where.first_tree_nodes;
            total += nodes[i];
        }
        std::vector<int32_t> par(static_cast<size_t>(total) + 1), tax(static_cast<size_t>(total) + 1);
        int rc = devforest_fetch_trees(ctx_, current(), count, first.data(), nodes.data(), par.data(), tax.data());
        if (rc) return rc;
        int64_t at = 0;
        std::vector<int32_t> where;
        for (int i = 0; i < count; ++i) {
            const int32_t slot = wave[single[i]].slot;
            where.assign(static_cast<size_t>(nodes[i]), 0);
            const bool shared = wave[single[i]].shared;
            where[0] = slot;
            set_taxon(slot, tax[at]);
            for (int64_t k = 1; k < nodes[i]; ++k) where[k] = add(where[par[at + k]], tax[at + k], shared);
            at += nodes[i];
        }
        return SCS_OK;
    }

    // ---- the three node paths, all on the wave's device-resident tours --------------------------------------------------
    int split_large(const Job &job, Split &s) {
        const DevForest &forest = current();
        const int n = static_cast<int>(job.taxa.size());
        const int T = job.where.trees;
        int rc;
        if ((rc = grow(ctx_, offsets_rel_, (static_cast<size_t>(T) + 1) * sizeof(int64_t)))) return rc;
        relative_offsets<<<ceil_div(T + 1, 256), 256, 0, ctx_->stream>>>(T + 1, forest.leaf_off.as<int64_t>() + job.where.tree_begin,
                                                                        offsets_rel_.as<int64_t>());
        SCS_LAUNCHED(ctx_, "relative_offsets");
        const int64_t L = job.leaves;
        ctx_->pending_units = static_cast<double>(job.where.pair_visits);
        ctx_->shard.engaged = job.shared;
        std::memset(&s.stats, 0, sizeof(s.stats));
        s.stats.eig[1] = s.stats.eig[2] = s.stats.residual = s.stats.margin = std::nan("");
        rc = node_split(ctx_, n, T, L, offsets_rel_.as<int64_t>(), tours_.leaf_taxon.as<int32_t>() + job.where.leaf_begin,
                        tours_.adj_depth.as<int32_t>() + job.where.leaf_begin, tours_.adj_val.as<double>() + job.where.leaf_begin,
                        tours_.root_depth.as<int32_t>() + job.where.tree_begin, forest.weight.as<double>() + job.where.tree_begin,
                        contract_, node_seed(seed_, job.taxa[0], job.taxa.size()), part_dev_.as<int32_t>() + s.part_at, nullptr,
                        &s.stats, true);
        ctx_->pending_units = 0.0;
        ctx_->shard.engaged = false;
        return rc;
    }

    int split_medium(scs_ctx *ctx, std::vector<Job> &wave, const std::vector<size_t> &medium, Split *splits,
                     std::vector<size_t> &reruns) {
        const DevForest &forest = current();
        const int B = static_cast<int>(medium.size());
        std::vector<int32_t> node_n(B), tree_begin(B), tree_end(B);
        std::vector<int64_t> part_off(B);
        std::vector<uint64_t> seeds(B);
        for (int b = 0; b < B; ++b) {
            const Job &job = wave[medium[b]];
            node_n[b] = static_cast<int32_t>(job.taxa.size());
            tree_begin[b] = job.where.tree_begin;
            tree_end[b] = job.where.tree_begin + job.where.trees;
            part_off[b] = splits[b].part_at;
            seeds[b] = node_seed(seed_, job.taxa[0], job.taxa.size());
        }
        std::vector<scs_node_stats> stats(B);
        std::vector<uint8_t> rerun(B, 0);
        int rc = medium_batch(ctx, B, node_n.data(), tree_begin.data(), tree_end.data(), part_off.data(), seeds.data(),
                              static_cast<int>(forest.trees), forest.leaves, forest.leaf_off.as<int64_t>(),
                              tours_.leaf_taxon.as<int32_t>(), tours_.adj_depth.as<int32_t>(), tours_.adj_val.as<double>(),
                              tours_.root_depth.as<int32_t>(), forest.weight.as<double>(), contract_, part_dev_.as<int32_t>(),
                              stats.data(), rerun.data());
        if (rc) return rc;
        for (int b = 0; b < B; ++b) {
            splits[b].stats = stats[b];
            if (rerun[b]) reruns.push_back(static_cast<size_t>(b));
        }
        return SCS_OK;
    }

    int split_small(scs_ctx *ctx, std::vector<Job> &wave, const std::vector<size_t> &small, Split *splits) {
        const DevForest &forest = current();
        const int B = static_cast<int>(small.size());
        std::vector<scs_small_node> desc(B);
        for (int b = 0; b < B; ++b) {
            const Job &job = wave[small[b]];
            desc[b].n = static_cast<int32_t>(job.taxa.size());
            desc[b].num_trees = job.where.trees;
            desc[b].leaf_base = job.where.leaf_begin;
            desc[b].tree_base = job.where.tree_begin;
            desc[b].vertex_base = splits[b].part_at;
        }
        int rc;
        const size_t bytes = sizeof(scs_small_node) * static_cast<size_t>(B);
        scs_small_node *desc_dev;
        if ((rc = reserve_as(ctx, SLOT_MED_NODES, static_cast<size_t>(B), &desc_dev))) return rc;
        void *pin_v;
        if ((rc = reserve_pinned(ctx, bytes + sizeof(scs_node_stats) * static_cast<size_t>(B) + 512, &pin_v))) return rc;
        unsigned char *pin = static_cast<unsigned char *>(pin_v);
        std::memcpy(pin, desc.data(), bytes);
        SCS_CUDA(ctx, cudaMemcpyAsync(desc_dev, pin, bytes, cudaMemcpyHostToDevice, ctx->stream));
        ctx->h2d_bytes += static_cast<int64_t>(bytes);
        scs_node_stats *stats_dev;
        if ((rc = reserve_as(ctx, SLOT_NODE_STATS, static_cast<size_t>(B), &stats_dev))) return rc;
        rc = small_batch(ctx, B, desc_dev, forest.leaf_off.as<int64_t>(), tours_.leaf_taxon.as<int32_t>(),
                         tours_.adj_depth.as<int32_t>(), tours_.adj_val.as<double>(), tours_.root_depth.as<int32_t>(),
                         forest.weight.as<double>(), contract_, part_dev_.as<int32_t>(), stats_dev, flags_dev_.as<int32_t>(), 1);
        if (rc) return rc;
        scs_node_stats *stats_pin = reinterpret_cast<scs_node_stats *>(pin + ((bytes + 255) & ~static_cast<size_t>(255)));
        SCS_CUDA(ctx, cudaMemcpyAsync(stats_pin, stats_dev, sizeof(scs_node_stats) * static_cast<size_t>(B), cudaMemcpyDeviceToHost,
                                       ctx->stream));
        SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        ctx->d2h_bytes += static_cast<int64_t>(sizeof(scs_node_stats)) * B;
        for (int b = 0; b < B; ++b) splits[b].stats = stats_pin[b];
        return SCS_OK;
    }

    // ---- what the split nodes turn into (scs.py:136-171): stars, sub-problems with restricted trees, singletons ---------
    int plan_children(std::vector<Job> &wave, std::vector<Split> &splits, std::vector<Job> &next) {
        const int J = static_cast<int>(wave.size());
        std::vector<int32_t> job_tree_begin(static_cast<size_t>(J) + 1, 0), job_parts(J, 0), job_part_base(J, 0);
        for (int j = 0; j < J; ++j) job_tree_begin[j] = wave[j].where.tree_begin;
        job_tree_begin[J] = static_cast<int32_t>(current().trees);
        std::sort(splits.begin(), splits.end(), [](const Split &a, const Split &b) { return a.job < b.job; });
        struct Pending {
            int32_t parent_slot;
            bool parent_shared, stays;     // the parent was a shared job; the child stays shared
            std::vector<int32_t> members;  // taxa of the component, ascending
        };
        std::vector<Pending> pending;      // one per new job
        std::vector<int32_t> part_newjob;  // global part -> new job or -1
        std::vector<int32_t> start, members, cursor;
        for (Split &s : splits) {
            const Job &job = wave[s.job];
            const std::vector<int32_t> &taxa = job.taxa;
            const int n = static_cast<int>(taxa.size());
            const int parts = s.stats.n_components != 1 ? s.stats.n_components : 2;
            const int32_t *part = part_.data() + s.part_at;
            if (record_) {
                scs_supertree::Record rec;
                rec.taxa = taxa;
                rec.part.assign(part, part + n);
                rec.stats = s.stats;
                rec.wave = static_cast<int32_t>(out_.waves - 1);
                (job.shared ? sh_records_ : out_.records).push_back(std::move(rec));
            }
            start.assign(parts + 1, 0);
            for (int v = 0; v < n; ++v) {
                if (part[v] < 0 || part[v] >= parts) return fail(ctx_, SCS_ERR_INVALID, "a partition label is out of range");
                start[part[v] + 1] += 1;
            }
            for (int c = 0; c < parts; ++c) start[c + 1] += start[c];
            members.resize(n);
            cursor.assign(start.begin(), start.end() - 1);
            for (int v = 0; v < n; ++v) members[cursor[part[v]]++] = taxa[v];
            s.parts = parts;
            s.part_base = static_cast<int32_t>(part_newjob.size());
            job_parts[s.job] = parts;
            job_part_base[s.job] = s.part_base;
            for (int c = 0; c < parts; ++c) {
                const int32_t *comp = members.data() + start[c];
                const int size = start[c + 1] - start[c];
                if (size == 0) {
                    part_newjob.push_back(-1);
                    continue;
                }
                // the children of a shared job are shared output nodes: every rank creates them, in the same order
                const int32_t child_slot = add(job.slot, -1, job.shared);
                if (size <= 2) {  // scs.py:143-145
                    fill_star(child_slot, comp, size, job.shared);
                    for (int i = 0; i < size; ++i) owner_[comp[i]] = -1;
                    part_newjob.push_back(-1);
                    continue;
                }
                bool stays = false;
                if (job.shared) {
                    stays = stays_shared(size);
                    if (!stays && deal(size) != rank_) {  // dealt to another rank: its owner restricts the trees to it
                        for (int i = 0; i < size; ++i) owner_[comp[i]] = -1;
                        part_newjob.push_back(-1);
                        continue;
                    }
                }
                const int32_t gp = static_cast<int32_t>(part_newjob.size());
                for (int i = 0; i < size; ++i) owner_[comp[i]] = gp;
                part_newjob.push_back(static_cast<int32_t>(pending.size()));
                pending.push_back(Pending{job.slot, job.shared, stays, std::vector<int32_t>(comp, comp + size)});
                pending_slot_.push_back(child_slot);
            }
        }
        const int new_jobs = static_cast<int>(pending.size());
        std::vector<DevJobInfo> info(static_cast<size_t>(new_jobs) + 1);
        if (new_jobs > 0) {
            Stopwatch sw_restrict(&restrict_device_s_);
            const int rc = devforest_restrict(ctx_, current(), J, job_tree_begin.data(), job_parts.data(), job_part_base.data(),
                                              static_cast<int>(part_newjob.size()), part_newjob.data(), new_jobs, owner_.data(),
                                              num_taxa_, &other(), info.data(), present_.data());
            if (rc) return rc;
        }
        // taxa of finished sub-problems keep no owner
        for (const Split &s : splits)
            for (int32_t x : wave[s.job].taxa) owner_[x] = -1;
        for (int j = 0; j < new_jobs; ++j) {
            Job child;
            child.slot = pending_slot_[j];
            child.where = info[j];
            // jobs are laid out in order: the leaves of a job end where the next job's begin
            child.leaves = (j + 1 < new_jobs ? info[j + 1].leaf_begin : other().leaves) - info[j].leaf_begin;
            // taxa of the component that are a tip of some kept tree; the others are attached as singleton children of
            // the parent (scs.py:168-171).  A child left without trees raises when its wave is processed.
            // (known to whoever restricted: to every rank only if the child stays shared)
            const bool empty = info[j].trees == 0;
            child.shared = pending[j].stays;
            for (int32_t x : pending[j].members) {
                if (present_[x]) child.taxa.push_back(x);
                else if (!empty) add(pending[j].parent_slot, x, pending[j].parent_shared && pending[j].stays);
            }
            next.push_back(std::move(child));
        }
        pending_slot_.clear();
        cur_ = cur_ < 0 ? 0 : 1 - cur_;
        return SCS_OK;
    }

    scs_ctx *ctx_;
    int weighting_, contract_;
    uint64_t seed_;
    bool record_;
    int rank_ = 0, world_ = 1;
    // Cooperative build over several GPUs (exchange windows connected, see driver.cu): a job of at least shard.min_n taxa
    // is SHARED -- every rank keeps its trees and the node is row-sharded over the GPUs; a smaller child of a shared
    // job is DEALT, with everything below it, to the rank with the least estimated work so far (every rank takes the
    // same decision from the same partition, nobody talks) and only its owner restricts the trees to it.  Shared
    // output nodes go to a list that is identical on every rank (ids <= -2) and becomes the shared prefix.
    bool cooperative_ = false;
    std::vector<double> load_;
    std::vector<int32_t> sh_parent_, sh_taxon_;
    std::vector<scs_supertree::Record> sh_records_;
    scs_supertree &out_;
    int num_taxa_ = 0;
    const DevForest *root_ = nullptr;  // the resident source trees (read-only): the forest of the first wave
    DriverCache &cache_;               // the context's buffers: they outlive the build
    DevForest (&forest_)[2];           // the forests of the later waves, written alternately
    int cur_ = -1;
    DevTours &tours_;
    GrowBuf &vertex_dev_, &offsets_rel_, &part_dev_, &flags_dev_;
    cudaEvent_t tours_ready_ = nullptr;
    std::vector<int32_t> vertex_, owner_, part_, pending_slot_;
    std::vector<uint8_t> present_;
    double restrict_device_s_ = 0.0;  // part of seconds[2] spent in devforest_restrict (launches + its round trips)
    const bool trace_ = std::getenv("SCS_DRIVER_TRACE") != nullptr;
};

}  // namespace

int run_device_driver(scs_ctx *ctx, const scs_device_forest *forest, int contract_edges, uint64_t seed, bool record, int rank,
                      int world, scs_supertree *out) {
    DeviceDriver driver(ctx, forest->weighting, contract_edges, seed, record, rank, world, out);
    return driver.run(forest);
}

}  // namespace scs

using namespace scs;

extern "C" {

int scs_device_forest_create(scs_ctx *ctx, const scs_forest *forest, int weighting, scs_device_forest **out) {
    return scs::device_forest_create(ctx, forest, weighting, false, out);
}

}  // extern "C"

// (re)fill a device forest object: its arrays only ever grow
static int device_forest_fill(scs_ctx *ctx, const scs_forest *forest, int weighting, bool cooperative, scs_device_forest *d) {
    d->weighting = weighting;
    d->num_taxa = scs_forest_num_taxa(forest);
    d->owner = ctx;
    d->taxa.clear();
    const int rc = devforest_upload(ctx, forest, weighting, &d->trees, cooperative);
    if (rc) return rc;
    std::vector<uint8_t> seen(static_cast<size_t>(d->num_taxa > 0 ? d->num_taxa : 1), 0);
    {
        const int32_t *tax = forest->taxon.data();
        const long long count = static_cast<long long>(forest->taxon.size());
        uint8_t *mark = seen.data();
#pragma omp parallel for schedule(static) num_threads(scs_host_threads() > 0 ? scs_host_threads() : 1) if (count > (1 << 20))
        for (long long k = 0; k < count; ++k)
            if (tax[k] >= 0) mark[tax[k]] = 1;  // racing writers all store 1
    }
    for (int x = 0; x < d->num_taxa; ++x)
        if (seen[x]) d->taxa.push_back(x);
    d->first_tree_nodes = forest->num_trees() > 0 ? forest->node_offsets[1] - forest->node_offsets[0] : 0;
    d->pair_visits = scs_forest_pair_visits(forest);
    d->leaves = forest->leaf_offsets.back();
    return SCS_OK;
}

int scs::device_forest_create(scs_ctx *ctx, const scs_forest *forest, int weighting, bool cooperative,
                              scs_device_forest **out) {
    if (!ctx || !forest || !out || weighting < 0 || weighting > 3) return SCS_ERR_INVALID;
    *out = nullptr;
    cudaSetDevice(ctx->device);
    scs_device_forest *d = new scs_device_forest();
    const int rc = device_forest_fill(ctx, forest, weighting, cooperative, d);
    if (rc) {
        d->trees.free_all(ctx);
        delete d;
        return rc;
    }
    *out = d;
    return SCS_OK;
}

// The device copy of the source trees scs_supertree_build works on: kept by the context between builds.
int scs::device_forest_refresh(scs_ctx *ctx, const scs_forest *forest, int weighting, bool cooperative,
                               const scs_device_forest **out) {
    if (!ctx || !forest || !out || weighting < 0 || weighting > 3) return SCS_ERR_INVALID;
    cudaSetDevice(ctx->device);
    scs_device_forest *d = &driver_cache(ctx).resident;
    *out = d;
    return device_forest_fill(ctx, forest, weighting, cooperative, d);
}

extern "C" {

int scs_device_forest_destroy(scs_device_forest *forest) {
    if (!forest) return SCS_OK;
    if (forest->owner) {
        cudaSetDevice(forest->owner->device);
        forest->trees.free_all(forest->owner);
        cudaStreamSynchronize(forest->owner->stream);
    }
    delete forest;
    return SCS_OK;
}

int64_t scs_device_forest_bytes(const scs_device_forest *forest) {
    if (!forest) return 0;
    const DevForest &f = forest->trees;
    return static_cast<int64_t>(2 * (f.trees + 1) * sizeof(int64_t) + f.nodes * 3 * sizeof(int32_t) +
                                (f.has_length ? f.nodes * sizeof(double) : 0) + (f.has_support ? f.nodes * sizeof(double) : 0) +
                                f.trees * (sizeof(double) + sizeof(int32_t)));
}

}  // extern "C"
