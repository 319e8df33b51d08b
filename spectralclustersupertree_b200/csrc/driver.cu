// The supertree recursion as a native work-list (host C++), feeding the GPU in waves.
//
// Restates the control flow of the reference's construct_supertree
// (/root/reference/src/sc_supertree/scs.py:96-174) over the flat forest store of forest.cpp:
// single-tree shortcut (:96-98), <= 2 names (:105-106), one recursion node on the GPU (:108-134),
// per component either a star (:143-145) or the restricted forest and a child task (:151-166), taxa
// that vanished from every restricted tree attached as singleton children (:168-171), children joined
// under a new root (:174).  Sub-problems are independent, so instead of recursing depth-first the
// driver processes the frontier breadth-first: all frontier nodes with <= 64 taxa (95 % of them on
// the 10 000-taxon workload) go to the GPU in ONE launch of small_batch_kernel with one host<->device
// round trip; larger nodes take the staged per-node path.
//
// The Python recursion in scs.py (supertree_of_forest) drives the same per-node entry points and is
// kept as the reference-shaped implementation; tests check the two produce the same supertree.

#include "common.cuh"

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <memory>
#include <thread>

#include <omp.h>

#include "forest.hpp"
#include "driver.hpp"

namespace scs {

namespace {

constexpr int kMaxWorkers = 16;       // upper bound on the contexts driving staged nodes concurrently
// how many of them are used (default 8; SCS_NODE_WORKERS overrides, for tuning)
int node_workers() {
    static const int value = [] {
        const char *env = std::getenv("SCS_NODE_WORKERS");
        const int v = env ? std::atoi(env) : 8;
        return v < 1 ? 1 : (v > kMaxWorkers ? kMaxWorkers : v);
    }();
    return value;
}
constexpr int kConcurrentMax = 4096;  // nodes above this many taxa run one at a time on the main context

struct Stopwatch {
    double *sink;
    std::chrono::steady_clock::time_point t0;
    explicit Stopwatch(double *s) : sink(s), t0(std::chrono::steady_clock::now()) {}
    ~Stopwatch() { *sink += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count(); }
};

struct Task {
    scs_forest *forest;
    bool owned;
    int32_t slot;                // output node this task fills in (node id: see Driver::add)
    std::vector<int32_t> taxa;   // taxa present in the forest, ascending (scs.py:708-725)
    bool shared = false;         // cooperative build: every rank processes this node (row-sharded over the GPUs)
};

// What one split recursion node turns into (scs.py:136-171), computed off the critical path.
enum ChildKind : int { CHILD_OWN = 0, CHILD_SHARED = 1, CHILD_DEALT_HERE = 2, CHILD_DEALT_AWAY = 3 };

struct Child {
    int kind = CHILD_OWN;          // cooperative build: who continues with this component
    std::vector<int32_t> star;     // <= 2 taxa: a tip or a star (scs.py:143-145) ...
    scs_forest *forest = nullptr;  // ... else the restricted forest of the component
    std::vector<int32_t> taxa;     // taxa present in that forest
    std::vector<int32_t> missing;  // taxa of the component in no restricted tree (scs.py:168-171)
};

struct SplitResult {
    size_t task = 0;
    std::vector<int32_t> part;
    scs_node_stats stats;
    std::vector<Child> children;
    int rc = SCS_OK;
};

// Per-thread scratch sized by the number of taxa of the job.
struct Scratch {
    std::vector<uint8_t> keep;
    std::vector<int32_t> stamp, local;
    int stamp_id = 0;
    void reset(int num_taxa) {
        keep.assign(num_taxa > 0 ? num_taxa : 1, 0);
        stamp.assign(num_taxa > 0 ? num_taxa : 1, 0);
        local.assign(num_taxa > 0 ? num_taxa : 1, -1);
        stamp_id = 0;
    }
    void present_taxa(const scs_forest *f, std::vector<int32_t> &taxa) {
        taxa.clear();
        ++stamp_id;
        for (int32_t x : f->taxon)
            if (x >= 0 && stamp[x] != stamp_id) {
                stamp[x] = stamp_id;
                taxa.push_back(x);
            }
        std::sort(taxa.begin(), taxa.end());
    }
};

// ---- a batch of small nodes from host memory: staging area + run -------------------------------------------
// The tours of the batch go through ONE pinned buffer and one H2D copy.  small_stage() sizes the buffer and
// says where each array lives in it, so the driver can flatten the tours straight into pinned memory;
// small_run() copies, launches small_batch_kernel and brings partitions and stats back.
struct SmallStage {
    size_t o_nodes = 0, o_off = 0, o_val = 0, o_w = 0, o_tax = 0, o_dep = 0, o_root = 0, total = 0;
    unsigned char *base = nullptr;  // pinned host memory
    scs_small_node *nodes() const { return reinterpret_cast<scs_small_node *>(base + o_nodes); }
    int64_t *off() const { return reinterpret_cast<int64_t *>(base + o_off); }
    double *val() const { return reinterpret_cast<double *>(base + o_val); }
    double *w() const { return reinterpret_cast<double *>(base + o_w); }
    int32_t *tax() const { return reinterpret_cast<int32_t *>(base + o_tax); }
    int32_t *dep() const { return reinterpret_cast<int32_t *>(base + o_dep); }
    int32_t *root() const { return reinterpret_cast<int32_t *>(base + o_root); }
};

int small_stage(scs_ctx *ctx, int num_nodes, int64_t L_total, int64_t T_total, SmallStage *st) {
    const size_t nB = static_cast<size_t>(num_nodes), nL = static_cast<size_t>(L_total), nT = static_cast<size_t>(T_total);
    st->o_nodes = 0;
    st->o_off = st->o_nodes + nB * sizeof(scs_small_node);
    st->o_val = st->o_off + (nT + nB) * sizeof(int64_t);
    st->o_w = st->o_val + nL * sizeof(double);
    st->o_tax = st->o_w + nT * sizeof(double);
    st->o_dep = st->o_tax + nL * sizeof(int32_t);
    st->o_root = st->o_dep + nL * sizeof(int32_t);
    st->total = st->o_root + nT * sizeof(int32_t) + 64;
    if (ctx->pinned_io_bytes < st->total) {
        if (ctx->pinned_io) {
            SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            SCS_CUDA(ctx, cudaFreeHost(ctx->pinned_io));
            ctx->pinned_io = nullptr;
            ctx->pinned_io_bytes = 0;
        }
        const size_t want = 2 * st->total + 4096;
        SCS_CUDA(ctx, cudaMallocHost(&ctx->pinned_io, want));
        ctx->pinned_io_bytes = want;
    }
    st->base = static_cast<unsigned char *>(ctx->pinned_io);
    return SCS_OK;
}

int small_run(scs_ctx *ctx, int num_nodes, const SmallStage &st, int contract_edges, int32_t *part,
              scs_node_stats *stats) {
    int64_t N_total = 0;
    const scs_small_node *nodes = st.nodes();
    for (int b = 0; b < num_nodes; ++b) {
        if (nodes[b].n < 1 || nodes[b].n > kSmallNode || nodes[b].num_trees < 0)
            return fail(ctx, SCS_ERR_INVALID, "small batch: node size out of range");
        if (nodes[b].num_trees > kSmallMaxTrees)
            return fail(ctx, SCS_ERR_INVALID, "small batch: more than 65 535 source trees at a node (use scs_node_split_*)");
        N_total += nodes[b].n;
    }
    const size_t nB = static_cast<size_t>(num_nodes);
    unsigned char *dev;
    int rc;
    if ((rc = reserve_as(ctx, SLOT_TOUR_OFFSETS, st.total, &dev))) return rc;
    SCS_CUDA(ctx, cudaMemcpyAsync(dev, st.base, st.total - 64, cudaMemcpyHostToDevice, ctx->stream));
    ctx->h2d_bytes += static_cast<int64_t>(st.total - 64);

    int32_t *part_dev, *bad_dev;
    scs_node_stats *stats_dev;
    if ((rc = reserve_as(ctx, SLOT_PART, static_cast<size_t>(N_total), &part_dev))) return rc;
    if ((rc = reserve_as(ctx, SLOT_NODE_STATS, nB, &stats_dev))) return rc;
    if ((rc = reserve_as(ctx, SLOT_SCALARS, 64, &bad_dev))) return rc;
    SCS_CUDA(ctx, cudaMemsetAsync(bad_dev, 0, sizeof(int32_t), ctx->stream));
    rc = small_batch(ctx, num_nodes, reinterpret_cast<const scs_small_node *>(dev + st.o_nodes),
                     reinterpret_cast<const int64_t *>(dev + st.o_off), reinterpret_cast<const int32_t *>(dev + st.o_tax),
                     reinterpret_cast<const int32_t *>(dev + st.o_dep), reinterpret_cast<const double *>(dev + st.o_val),
                     reinterpret_cast<const int32_t *>(dev + st.o_root), reinterpret_cast<const double *>(dev + st.o_w),
                     contract_edges, part_dev, stats_dev, bad_dev);
    if (rc) return rc;
    void *pin_v;
    if ((rc = reserve_pinned(ctx, 64, &pin_v))) return rc;
    SCS_CUDA(ctx, cudaMemcpyAsync(part, part_dev, sizeof(int32_t) * N_total, cudaMemcpyDeviceToHost, ctx->stream));
    SCS_CUDA(ctx, cudaMemcpyAsync(stats, stats_dev, sizeof(scs_node_stats) * nB, cudaMemcpyDeviceToHost, ctx->stream));
    SCS_CUDA(ctx, cudaMemcpyAsync(pin_v, bad_dev, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->d2h_bytes += static_cast<int64_t>(sizeof(int32_t) * N_total + sizeof(scs_node_stats) * nB);
    if (*static_cast<int32_t *>(pin_v) != 0) return fail(ctx, SCS_ERR_INPUT, "leaf tour: taxon id out of range");
    for (int b = 0; b < num_nodes; ++b)
        if (stats[b].solver == -1) {
            stats[b].solver = 0;
            return fail(ctx, SCS_ERR_TOO_SMALL, "spectral step on a graph contracted to one vertex");
        }
    return SCS_OK;
}

class Driver {
  public:
    Driver(scs_ctx *ctx, int weighting, int contract_edges, uint64_t seed, bool record, int rank, int world,
           scs_supertree *out)
        : ctx_(ctx), weighting_(weighting), contract_(contract_edges), seed_(seed), record_(record), rank_(rank),
          world_(world), out_(*out) {}

    int run(const scs_forest *root) {
        num_taxa_ = scs_forest_num_taxa(root);
        scratch_.resize(static_cast<size_t>(std::max(scs_host_threads(), kMaxWorkers)));
        for (Scratch &sc : scratch_) sc.reset(num_taxa_);
        std::vector<Task> wave, next;
        // While all ranks still walk the same frontier, nodes large enough are shared out over the GPUs
        // (shard.cu).  Cooperative build (exchange windows connected): see the comment at stays_shared().
        const ShardState &sh = ctx_->shard;
        cooperative_ = world_ > 1 && sh.connected && sh.world == world_ && sh.rank == rank_;
        ctx_->shard.engaged = cooperative_;
        const int32_t root_slot = add(-1, -1, cooperative_);
        wave.push_back(Task{const_cast<scs_forest *>(root), false, root_slot, {}});
        scratch_[0].present_taxa(root, wave[0].taxa);
        if (cooperative_) {
            load_.assign(static_cast<size_t>(world_), 0.0);
            const int n_root = static_cast<int>(wave[0].taxa.size());
            wave[0].shared = stays_shared(n_root);
            if (!wave[0].shared && deal(n_root) != rank_) wave.clear();  // a small job: one rank does it all
        }
        int rc = SCS_OK;
        bool shared_phase = cooperative_;
        while (rc == SCS_OK) {
            if (wave.empty()) {
                if (!shared_phase) break;
                // the shared frontier is exhausted: from here on this rank works through its own backlog alone
                shared_phase = false;
                ctx_->shard.engaged = false;
                wave.swap(backlog_);
                if (wave.empty()) break;
            }
            if (world_ > 1 && !cooperative_ && !partitioned_ && should_partition(wave)) partition(wave);
            if (wave.empty()) break;
            out_.waves += 1;
            int32_t max_n = 0;
            for (const Task &t : wave) max_n = std::max<int32_t>(max_n, static_cast<int32_t>(t.taxa.size()));
            out_.wave_tasks.push_back(static_cast<int32_t>(wave.size()));
            out_.wave_max_n.push_back(max_n);
            next.clear();
            const double before_gpu = out_.seconds[0] + out_.seconds[1] + out_.medium_seconds, before_restrict = out_.seconds[2];
            const auto wave_start = std::chrono::steady_clock::now();
            rc = process_wave(wave, next);
            out_.wave_seconds.push_back(out_.seconds[0] + out_.seconds[1] + out_.medium_seconds - before_gpu);
            out_.wave_seconds.push_back(out_.seconds[2] - before_restrict);
            out_.wave_seconds.push_back(std::chrono::duration<double>(std::chrono::steady_clock::now() - wave_start).count());
            const auto t_destroy = std::chrono::steady_clock::now();
            for (Task &t : wave)
                if (t.owned) scs_forest_destroy(t.forest);
            if (trace_) {
                const double destroy = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_destroy).count();
                std::fprintf(stderr, "[scs driver] wave %d: tasks %zu, induce %.2f ms, present_taxa %.2f ms, destroy %.2f ms\n",
                             static_cast<int>(out_.waves), wave.size(), 1e3 * trace_induce_, 1e3 * trace_present_, 1e3 * destroy);
                trace_induce_ = trace_present_ = 0.0;
            }
            wave.clear();
            wave.swap(next);
        }
        for (Task &t : wave)  // only non-empty after an error: the sub-problems that were never started
            if (t.owned) scs_forest_destroy(t.forest);
        for (Task &t : backlog_)
            if (t.owned) scs_forest_destroy(t.forest);
        backlog_.clear();
        ctx_->shard.engaged = false;
        if (rc == SCS_OK && cooperative_) finish_cooperative();
        return rc;
    }

  private:
    // ---- sharding over ranks (one process per GPU) ----------------------------------------------------
    // Sub-problems are independent (scs.py:139-166), so one job is spread over GPUs by giving each rank
    // a share of the frontier.  Every rank runs the first waves redundantly -- the kernels are
    // deterministic, so all ranks hold the same frontier and the same output prefix without talking --
    // until the frontier is wide enough; then the frontier is dealt out (largest estimated cost first,
    // to the least loaded rank) and each rank finishes only its own sub-problems.  The caller
    // concatenates the ranks' outputs past the shared prefix (no collective on the data path).
    // ---- output nodes ------------------------------------------------------------------------------------
    // Node ids: id >= 0 is a node of this rank's own list (out_.parent / out_.taxon); id <= -2 is node -2 - id of
    // the shared list, which only exists in a cooperative build and is identical on every rank (except for a
    // taxon its owner writes into a dealt slot).  -1 is "no parent".
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

    // ref: scs.py:728-746 + _connect_trees :390-408 -- one name stays a tip, more become a star
    void fill_star(int32_t slot, const int32_t *taxa, int count, bool shared) {
        if (count == 1) {
            set_taxon(slot, taxa[0]);
            return;
        }
        for (int i = 0; i < count; ++i) add(slot, taxa[i], shared);
    }

    // topology-only copy of the single remaining tree (ref: scs.py:96-98)
    int fill_tree(int32_t slot, const scs_forest *f, bool shared) {
        int64_t count = 0;
        int rc = scs_forest_tree_info(f, 0, &count, nullptr, nullptr);
        if (rc) return rc;
        std::vector<int32_t> par(count), tax(count), where(count);
        if ((rc = scs_forest_tree(f, 0, par.data(), nullptr, nullptr, tax.data()))) return rc;
        where[0] = slot;
        set_taxon(slot, tax[0]);
        for (int64_t k = 1; k < count; ++k) where[k] = add(where[par[k]], tax[k], shared);
        return SCS_OK;
    }

    // ---- cooperative build (exchange windows connected) -----------------------------------------------------
    // A component of at least shard.min_n taxa stays SHARED: every rank keeps its forest and the node is
    // row-sharded over the GPUs.  A smaller component is DEALT at once, with everything below it, to the
    // rank with the least estimated work so far (every rank takes the same decision from the same partition,
    // nobody talks); only its owner restricts the source trees to it.  Ranks first walk the shared frontier in
    // lock-step, wave by wave, putting what is dealt to them on a backlog, and then work through the backlog
    // alone.  Shared nodes go to a list that is identical on every rank and becomes the shared prefix of the
    // output; the caller joins the ranks' outputs as in the non-cooperative build.
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

    static double task_cost(const Task &t) {
        const double n = static_cast<double>(t.taxa.size());
        return static_cast<double>(scs_forest_pair_visits(t.forest)) + 64.0 * n * n + 2.0e4;
    }

    bool should_partition(const std::vector<Task> &wave) const {
        if (static_cast<int>(wave.size()) >= 8 * world_) return true;
        // or: the frontier can already be balanced to within ~20 % of an even share
        if (static_cast<int>(wave.size()) < world_) return false;
        double total = 0.0, largest = 0.0;
        for (const Task &t : wave) {
            const double c = task_cost(t);
            total += c;
            largest = std::max(largest, c);
        }
        return largest <= 1.2 * total / world_;
    }

    void partition(std::vector<Task> &wave) {
        partitioned_ = true;
        ctx_->shard.engaged = false;
        out_.shared_prefix = static_cast<int64_t>(out_.parent.size());
        std::vector<size_t> order(wave.size());
        for (size_t i = 0; i < order.size(); ++i) order[i] = i;
        std::vector<double> cost(wave.size());
        for (size_t i = 0; i < wave.size(); ++i) cost[i] = task_cost(wave[i]);
        std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return cost[a] > cost[b]; });
        std::vector<double> load(world_, 0.0);
        std::vector<int> owner(wave.size(), 0);
        for (size_t i : order) {
            const int r = static_cast<int>(std::min_element(load.begin(), load.end()) - load.begin());
            owner[i] = r;
            load[r] += cost[i];
        }
        std::vector<Task> mine;
        for (size_t i = 0; i < wave.size(); ++i) {
            if (owner[i] == rank_) mine.push_back(std::move(wave[i]));
            else if (wave[i].owned) scs_forest_destroy(wave[i].forest);
        }
        wave.swap(mine);
    }

    int process_wave(std::vector<Task> &wave, std::vector<Task> &next) {
        std::vector<size_t> small, medium;
        std::vector<SplitResult> results;
        int rc;
        for (size_t i = 0; i < wave.size(); ++i) {
            Task &task = wave[i];
            const int T = scs_forest_num_trees(task.forest);
            if (T == 0) return fail(ctx_, SCS_ERR_EMPTY, "a component is covered by no source tree (scs.py:63-65)");
            if (T == 1) {
                if ((rc = fill_tree(task.slot, task.forest, task.shared))) return rc;
                continue;
            }
            const int n = static_cast<int>(task.taxa.size());
            if (n <= 2) {
                fill_star(task.slot, task.taxa.data(), n, task.shared);
                continue;
            }
            if (n <= ctx_->small_limit && T <= kSmallMaxTrees) {
                small.push_back(i);
                continue;
            }
            if (n <= ctx_->medium_limit && !shard_applies(ctx_, n)) {
                medium.push_back(i);
                continue;
            }
            results.emplace_back();
            results.back().task = i;
        }
        // The three kinds of nodes of a wave run next to each other: the batch of small nodes and the batch of
        // medium nodes each on its own context (stream) and host thread, the large nodes on this thread.
        {
            std::vector<SplitResult> small_results, medium_results;
            int small_rc = SCS_OK, medium_rc = SCS_OK;
            const bool busy_here = !results.empty();
            const bool small_aside = !small.empty() && (busy_here || !medium.empty()) && small_context() != nullptr;
            const bool medium_aside = !medium.empty() && busy_here && medium_context() != nullptr;
            std::thread small_thread, medium_thread;
            if (small_aside)
                small_thread = std::thread([&] {
                    const cudaError_t err = cudaSetDevice(ctx_->device);
                    small_rc = err != cudaSuccess ? fail(small_ctx_, SCS_ERR_CUDA, "cudaSetDevice (small-node thread)", err)
                                                  : split_small(small_ctx_, scratch_small_, wave, small, small_results);
                });
            if (medium_aside)
                medium_thread = std::thread([&] {
                    const cudaError_t err = cudaSetDevice(ctx_->device);
                    medium_rc = err != cudaSuccess ? fail(medium_ctx_, SCS_ERR_CUDA, "cudaSetDevice (medium-node thread)", err)
                                                   : split_medium(medium_ctx_, scratch_medium_, wave, medium, medium_results);
                });
            rc = split_large_all(wave, results);
            if (rc == SCS_OK && !medium.empty() && !medium_aside) rc = split_medium(ctx_, scratch_, wave, medium, results);
            if (rc == SCS_OK && !small.empty() && !small_aside) rc = split_small(ctx_, scratch_, wave, small, results);
            if (small_thread.joinable()) small_thread.join();
            if (medium_thread.joinable()) medium_thread.join();
            if (small_aside) fold_counters(small_ctx_);
            if (medium_aside) fold_counters(medium_ctx_);
            out_.medium_seconds += medium_seconds_ - medium_tour_seconds_;
            out_.seconds[3] += medium_tour_seconds_;
            medium_seconds_ = medium_tour_seconds_ = 0.0;
            if (rc == SCS_OK && small_rc != SCS_OK) {
                ctx_->last_error = small_ctx_->last_error;
                rc = small_rc;
            }
            if (rc == SCS_OK && medium_rc != SCS_OK) {
                ctx_->last_error = medium_ctx_->last_error;
                rc = medium_rc;
            }
            if (rc) return rc;
            for (SplitResult &res : medium_results) results.push_back(std::move(res));
            for (SplitResult &res : small_results) results.push_back(std::move(res));
        }

        // children of every split node (scs.py:136-171).  The restrictions of the whole wave run as ONE
        // batch over all host threads: (child, source tree) pairs are the work items, so a wave of two huge
        // restrictions is spread as evenly as one of a thousand small ones.
        {
            Stopwatch sw(&out_.seconds[2]);
            if ((rc = plan_wave(wave, results))) {
                for (SplitResult &res : results)
                    for (Child &child : res.children)
                        if (child.forest) scs_forest_destroy(child.forest);
                return rc;
            }
        }
        for (SplitResult &res : results) emit(wave[res.task], res, next);
        return SCS_OK;
    }

    // local[] maps global taxon id -> vertex id of the node; only the node's own taxa are ever read
    int tours_of(const scs_forest *f, const std::vector<int32_t> &taxa, std::vector<int32_t> &local,
                 int64_t *leaf_offsets, int32_t *leaf_taxon, int32_t *adj_depth, double *adj_val, int32_t *root_depth,
                 double *tree_weight) {
        for (size_t v = 0; v < taxa.size(); ++v) local[taxa[v]] = static_cast<int32_t>(v);
        return scs_forest_tours(f, weighting_, local.data(), leaf_offsets, leaf_taxon, adj_depth, adj_val, root_depth,
                                tree_weight);
    }

    // Host buffers for one node's tours (one set per worker).
    struct TourBuffers {
        std::vector<int64_t> off;
        std::vector<int32_t> tax, dep, root;
        std::vector<double> val, wgt;
    };

    int split_large(scs_ctx *ctx, TourBuffers &buf, Scratch &scratch, Task &task, SplitResult &res) {
        const scs_forest *f = task.forest;
        const std::vector<int32_t> &taxa = task.taxa;
        const int n = static_cast<int>(taxa.size());
        const int T = scs_forest_num_trees(f);
        const int64_t L = scs_forest_num_leaves(f);
        buf.off.resize(T + 1);
        buf.tax.resize(L + 1);
        buf.dep.resize(L + 1);
        buf.val.resize(L + 1);
        buf.root.resize(T + 1);
        buf.wgt.resize(T + 1);
        int rc = tours_of(f, taxa, scratch.local, buf.off.data(), buf.tax.data(), buf.dep.data(), buf.val.data(),
                          buf.root.data(), buf.wgt.data());
        if (rc) return rc;
        res.part.resize(n);
        // the seed only picks the Lanczos start vector; it is a function of the node's taxa (driver.hpp)
        return node_split_host(ctx, n, T, L, buf.off.data(), buf.tax.data(), buf.dep.data(), buf.val.data(),
                               buf.root.data(), buf.wgt.data(), contract_, node_seed(seed_, taxa[0], taxa.size()),
                               res.part.data(), &res.stats, true);
    }

    // The staged path is a chain of small launches and a few host round trips per node: latency, not
    // throughput.  Nodes of one wave are independent, so those that fit a worker's workspace are driven
    // by several host threads at once, each with its own context (stream + workspace) on the same GPU;
    // the GPU overlaps their kernels.  The few very large nodes stay on the main context, one at a time.
    int split_large_all(std::vector<Task> &wave, std::vector<SplitResult> &results) {
        if (results.empty()) return SCS_OK;
        Stopwatch sw(&out_.seconds[0]);
        std::vector<int> serial, concurrent;
        for (int r = 0; r < static_cast<int>(results.size()); ++r) {
            const Task &task = wave[results[r].task];
            {
                const int64_t visits = scs_forest_pair_visits(task.forest);
#pragma omp atomic
                out_.pair_visits += visits;
            }
            const int n = static_cast<int>(task.taxa.size());
            (n > kConcurrentMax || shard_applies(ctx_, n) ? serial : concurrent).push_back(r);
        }
        out_.nodes_large += static_cast<int64_t>(results.size());
        if (buffers_.empty()) buffers_.resize(1);
        for (int r : serial) {
            const int rc = split_large(ctx_, buffers_[0], scratch_[0], wave[results[r].task], results[r]);
            if (rc) return rc;
        }
        const int jobs = static_cast<int>(concurrent.size());
        if (jobs == 0) return SCS_OK;
        const int workers = std::max(1, std::min({node_workers(), jobs, scs_host_threads()}));
        int rc = ensure_workers(ctx_, workers);
        if (rc) return rc;
        if (static_cast<int>(buffers_.size()) < workers) buffers_.resize(workers);
        {
            // any worker may draw the largest node of the wave: size them all for it now
            int big_n = 0, big_T = 0;
            int64_t big_L = 0;
            for (int r : concurrent) {
                const Task &task = wave[results[r].task];
                big_n = std::max(big_n, static_cast<int>(task.taxa.size()));
                big_T = std::max(big_T, scs_forest_num_trees(task.forest));
                big_L = std::max<int64_t>(big_L, scs_forest_num_leaves(task.forest));
            }
            for (int w = 0; w < workers; ++w)
                if ((rc = prewarm_node(w == 0 ? ctx_ : ctx_->workers[w - 1], big_n, big_T, big_L))) return rc;
        }
        int first_error = SCS_OK;
#pragma omp parallel for schedule(dynamic, 1) num_threads(workers) if (workers > 1)
        for (int i = 0; i < jobs; ++i) {
            const int w = omp_get_thread_num();
            scs_ctx *ctx = w == 0 ? ctx_ : ctx_->workers[w - 1];
            SplitResult &res = results[concurrent[i]];
            const cudaError_t dev_err = cudaSetDevice(ctx->device);
            const int status = dev_err != cudaSuccess
                                   ? fail(ctx, SCS_ERR_CUDA, "cudaSetDevice (node worker thread)", dev_err)
                                   : split_large(ctx, buffers_[w], scratch_[w], wave[res.task], res);
            if (status) {
                if (ctx != ctx_) ctx_->last_error = ctx->last_error;
#pragma omp atomic write
                first_error = status;
            }
        }
        for (scs_ctx *worker : ctx_->workers) fold_counters(worker);
        return first_error;
    }

    // fold another context's counters into the main context
    void fold_counters(scs_ctx *other) {
        ctx_->launches += other->launches;
        ctx_->h2d_bytes += other->h2d_bytes;
        ctx_->d2h_bytes += other->d2h_bytes;
        other->launches = 0;
        other->h2d_bytes = other->d2h_bytes = 0;
        for (int k = 0; k < 8; ++k) {
            ctx_->stage_seconds[k] += other->stage_seconds[k];
            other->stage_seconds[k] = 0.0;
        }
    }

    // The context the batch of small nodes uses when it runs next to the large nodes (the last worker slot).
    scs_ctx *small_context() {
        if (small_ctx_) return small_ctx_;
        if (scs_host_threads() < 2) return nullptr;
        if (ensure_workers(ctx_, kMaxWorkers + 1) != SCS_OK) return nullptr;
        small_ctx_ = ctx_->workers[kMaxWorkers - 1];
        small_ctx_->small_limit = ctx_->small_limit;
        scratch_small_.resize(scratch_.size());
        for (Scratch &sc : scratch_small_) sc.reset(num_taxa_);
        return small_ctx_;
    }

    // The context of the batch of medium nodes when it runs next to the large nodes (the last worker slot but one).
    scs_ctx *medium_context() {
        if (medium_ctx_) return medium_ctx_;
        if (scs_host_threads() < 2) return nullptr;
        if (ensure_workers(ctx_, kMaxWorkers + 1) != SCS_OK) return nullptr;
        medium_ctx_ = ctx_->workers[kMaxWorkers - 2];
        scratch_medium_.resize(scratch_.size());
        for (Scratch &sc : scratch_medium_) sc.reset(num_taxa_);
        return medium_ctx_;
    }

    // All nodes of a wave between the small-node limit and the medium-node limit in one batch (csrc/medium.cu): their
    // tours are flattened into one pinned staging area (absolute leaf offsets), copied in one piece, and every
    // stage of the node path is one launch over the whole batch.
    int split_medium(scs_ctx *ctx, std::vector<Scratch> &scratch, std::vector<Task> &wave,
                     const std::vector<size_t> &medium, std::vector<SplitResult> &results) {
        const int B = static_cast<int>(medium.size());
        Stopwatch sw_all(&medium_seconds_);  // merged into the totals after the wave's threads are joined
        std::vector<int32_t> node_n(B), tree_begin(B + 1, 0);
        std::vector<int64_t> leaf_base(B + 1, 0), part_off(B + 1, 0);
        std::vector<uint64_t> seeds(B);
        int64_t visits = 0;
        for (int b = 0; b < B; ++b) {
            const Task &task = wave[medium[b]];
            node_n[b] = static_cast<int32_t>(task.taxa.size());
            tree_begin[b + 1] = tree_begin[b] + scs_forest_num_trees(task.forest);
            leaf_base[b + 1] = leaf_base[b] + scs_forest_num_leaves(task.forest);
            part_off[b + 1] = part_off[b] + node_n[b];
            seeds[b] = node_seed(seed_, task.taxa[0], task.taxa.size());
            visits += scs_forest_pair_visits(task.forest);
        }
        {
#pragma omp atomic
            out_.pair_visits += visits;
        }
        const size_t nT = static_cast<size_t>(tree_begin[B]), nL = static_cast<size_t>(leaf_base[B]);
        // staging layout: offsets | values | weights | taxa | depths | root depths
        const size_t o_off = 0, o_val = o_off + (nT + 1) * sizeof(int64_t), o_w = o_val + nL * sizeof(double),
                     o_tax = o_w + nT * sizeof(double), o_dep = o_tax + nL * sizeof(int32_t),
                     o_root = o_dep + nL * sizeof(int32_t), total = o_root + nT * sizeof(int32_t) + 64;
        if (ctx->pinned_io_bytes < total) {
            if (ctx->pinned_io) {
                SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
                SCS_CUDA(ctx, cudaFreeHost(ctx->pinned_io));
                ctx->pinned_io = nullptr;
                ctx->pinned_io_bytes = 0;
            }
            const size_t want = 2 * total + 4096;
            SCS_CUDA(ctx, cudaMallocHost(&ctx->pinned_io, want));
            ctx->pinned_io_bytes = want;
        }
        unsigned char *stage = static_cast<unsigned char *>(ctx->pinned_io);
        int64_t *s_off = reinterpret_cast<int64_t *>(stage + o_off);
        double *s_val = reinterpret_cast<double *>(stage + o_val), *s_w = reinterpret_cast<double *>(stage + o_w);
        int32_t *s_tax = reinterpret_cast<int32_t *>(stage + o_tax), *s_dep = reinterpret_cast<int32_t *>(stage + o_dep),
                *s_root = reinterpret_cast<int32_t *>(stage + o_root);
        int tours_rc = SCS_OK;
        const int tour_threads = ctx == ctx_ ? scs_host_threads() : std::max(1, scs_host_threads() / 2);
        {
            Stopwatch sw(&medium_tour_seconds_);
#pragma omp parallel num_threads(tour_threads) if (B >= 2)
            {
                std::vector<int64_t> own_off;
#pragma omp for schedule(dynamic, 1)
                for (int b = 0; b < B; ++b) {
                    const Task &task = wave[medium[b]];
                    const int T = tree_begin[b + 1] - tree_begin[b];
                    own_off.resize(static_cast<size_t>(T) + 1);
                    const int status = tours_of(task.forest, task.taxa, scratch[static_cast<size_t>(omp_get_thread_num())].local,
                                                own_off.data(), s_tax + leaf_base[b], s_dep + leaf_base[b], s_val + leaf_base[b],
                                                s_root + tree_begin[b], s_w + tree_begin[b]);
                    for (int t = 0; t < T; ++t) s_off[tree_begin[b] + t] = leaf_base[b] + own_off[t];
                    if (status) {
#pragma omp atomic write
                        tours_rc = status;
                    }
                }
            }
            s_off[nT] = leaf_base[B];
        }
        if (tours_rc) return tours_rc;
        unsigned char *dev;
        int rc;
        if ((rc = reserve_as(ctx, SLOT_TOUR_OFFSETS, total, &dev))) return rc;
        SCS_CUDA(ctx, cudaMemcpyAsync(dev, stage, total - 64, cudaMemcpyHostToDevice, ctx->stream));
        ctx->h2d_bytes += static_cast<int64_t>(total - 64);
        int32_t *part_dev;
        if ((rc = reserve_as(ctx, SLOT_PART, static_cast<size_t>(part_off[B]) + 1, &part_dev))) return rc;
        std::vector<scs_node_stats> stats(B);
        std::vector<uint8_t> rerun(B, 0);
        rc = medium_batch(ctx, B, node_n.data(), tree_begin.data(), tree_begin.data() + 1, part_off.data(), seeds.data(), static_cast<int>(nT),
                          static_cast<int64_t>(nL), reinterpret_cast<const int64_t *>(dev + o_off),
                          reinterpret_cast<const int32_t *>(dev + o_tax), reinterpret_cast<const int32_t *>(dev + o_dep),
                          reinterpret_cast<const double *>(dev + o_val), reinterpret_cast<const int32_t *>(dev + o_root),
                          reinterpret_cast<const double *>(dev + o_w), contract_, part_dev, stats.data(), rerun.data());
        if (rc) return rc;
        std::vector<int32_t> part(static_cast<size_t>(part_off[B]) + 1);
        SCS_CUDA(ctx, cudaMemcpyAsync(part.data(), part_dev, sizeof(int32_t) * part_off[B], cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        ctx->d2h_bytes += static_cast<int64_t>(sizeof(int32_t)) * part_off[B];
        out_.nodes_medium += B;
        if (medium_buffers_.empty()) medium_buffers_.resize(1);
        for (int b = 0; b < B; ++b) {
            results.emplace_back();
            SplitResult &res = results.back();
            res.task = medium[b];
            if (rerun[b]) {
                // eigensolver restart / repeated-eigenvalue check: the per-node path has both
                out_.nodes_rerun += 1;
                if ((rc = split_large(ctx, medium_buffers_[0], scratch[0], wave[medium[b]], res))) return rc;
                continue;
            }
            res.part.assign(part.data() + part_off[b], part.data() + part_off[b + 1]);
            res.stats = stats[b];
        }
        return SCS_OK;
    }

    int split_small(scs_ctx *ctx, std::vector<Scratch> &scratch, std::vector<Task> &wave,
                    const std::vector<size_t> &small, std::vector<SplitResult> &results) {
        const int B = static_cast<int>(small.size());
        int64_t visits = 0;
        std::vector<scs_small_node> nodes(B);
        int64_t L_total = 0, T_total = 0, N_total = 0;
        for (int b = 0; b < B; ++b) {
            const scs_forest *f = wave[small[b]].forest;
            nodes[b].n = static_cast<int32_t>(wave[small[b]].taxa.size());
            nodes[b].num_trees = scs_forest_num_trees(f);
            nodes[b].leaf_base = L_total;
            nodes[b].tree_base = T_total;
            nodes[b].vertex_base = N_total;
            L_total += scs_forest_num_leaves(f);
            T_total += nodes[b].num_trees;
            N_total += nodes[b].n;
            visits += scs_forest_pair_visits(f);
        }
        {
#pragma omp atomic
            out_.pair_visits += visits;
        }
        // the tours are flattened straight into the pinned staging area of the batch
        SmallStage stage;
        int rc = small_stage(ctx, B, L_total, T_total, &stage);
        if (rc) return rc;
        std::memcpy(stage.nodes(), nodes.data(), sizeof(scs_small_node) * static_cast<size_t>(B));
        int tours_rc = SCS_OK;
        // next to the large nodes (own context) the host threads are shared with their workers: a small team
        const int tour_threads = ctx == ctx_ ? scs_host_threads() : std::max(1, std::min(4, scs_host_threads() / 4));
        {
            Stopwatch sw(&out_.seconds[3]);
#pragma omp parallel for schedule(dynamic, 8) if (B >= 32) num_threads(tour_threads)
            for (int b = 0; b < B; ++b) {
                const scs_forest *f = wave[small[b]].forest;
                const int status = tours_of(f, wave[small[b]].taxa, scratch[static_cast<size_t>(omp_get_thread_num())].local,
                                            stage.off() + nodes[b].tree_base + b, stage.tax() + nodes[b].leaf_base,
                                            stage.dep() + nodes[b].leaf_base, stage.val() + nodes[b].leaf_base,
                                            stage.root() + nodes[b].tree_base, stage.w() + nodes[b].tree_base);
                if (status) {
#pragma omp atomic write
                    tours_rc = status;
                }
            }
        }
        if (tours_rc) return tours_rc;
        part_.resize(N_total);
        std::vector<scs_node_stats> stats(B);
        {
            Stopwatch sw(&out_.seconds[1]);
            rc = small_run(ctx, B, stage, contract_, part_.data(), stats.data());
        }
        if (rc) return rc;
        out_.nodes_small += B;
        for (int b = 0; b < B; ++b) {
            results.emplace_back();
            SplitResult &res = results.back();
            res.task = small[b];
            res.part.assign(part_.data() + nodes[b].vertex_base, part_.data() + nodes[b].vertex_base + nodes[b].n);
            res.stats = stats[b];
        }
        return SCS_OK;
    }

    // ref: scs.py:136-171 -- what the children of the split nodes of a wave are
    int plan_wave(const std::vector<Task> &wave, std::vector<SplitResult> &results) {
        struct Pending {
            SplitResult *res;
            size_t child;       // index into res->children
            std::vector<int32_t> members;  // taxa of the component, ascending
        };
        std::vector<Pending> pending;
        std::vector<scs_induce_job> jobs;
        if (owner_.size() < static_cast<size_t>(num_taxa_)) owner_.assign(static_cast<size_t>(num_taxa_), -1);
        if (present_.size() < static_cast<size_t>(num_taxa_)) present_.assign(static_cast<size_t>(num_taxa_), 0);
        std::vector<int32_t> start, members, cursor;
        for (SplitResult &res : results) {
            const Task &task = wave[res.task];
            const std::vector<int32_t> &taxa = task.taxa;
            const int n = static_cast<int>(taxa.size());
            const int parts = res.stats.n_components != 1 ? res.stats.n_components : 2;
            const int32_t *part = res.part.data();
            // bucket the vertices by part, keeping ascending taxon order inside each
            start.assign(parts + 1, 0);
            for (int v = 0; v < n; ++v) {
                if (part[v] < 0 || part[v] >= parts) return fail(ctx_, SCS_ERR_INVALID, "a partition label is out of range");
                start[part[v] + 1] += 1;
            }
            for (int c = 0; c < parts; ++c) start[c + 1] += start[c];
            members.resize(n);
            cursor.assign(start.begin(), start.end() - 1);
            for (int v = 0; v < n; ++v) members[cursor[part[v]]++] = taxa[v];
            for (int c = 0; c < parts; ++c) {
                const int32_t *comp = members.data() + start[c];
                const int size = start[c + 1] - start[c];
                if (size == 0) continue;
                res.children.emplace_back();
                Child &child = res.children.back();
                if (size <= 2) {  // ref: scs.py:143-145
                    child.star.assign(comp, comp + size);
                    for (int i = 0; i < size; ++i) owner_[comp[i]] = -1;
                    continue;
                }
                if (task.shared) {
                    child.kind = stays_shared(size) ? CHILD_SHARED : (deal(size) == rank_ ? CHILD_DEALT_HERE : CHILD_DEALT_AWAY);
                    if (child.kind == CHILD_DEALT_AWAY) {  // its owner restricts the trees to it
                        for (int i = 0; i < size; ++i) owner_[comp[i]] = -1;
                        continue;
                    }
                }
                const int32_t job = static_cast<int32_t>(jobs.size());
                for (int i = 0; i < size; ++i) owner_[comp[i]] = job;
                scs_induce_job spec;
                spec.src = task.forest;
                jobs.push_back(spec);
                pending.push_back(Pending{&res, res.children.size() - 1, std::vector<int32_t>(comp, comp + size)});
            }
        }
        const auto t_induce = std::chrono::steady_clock::now();
        const int rc = scs_forest_induce_batch(jobs.data(), static_cast<int>(jobs.size()), owner_.data(), present_.data());
        if (trace_) trace_induce_ += std::chrono::duration<double>(std::chrono::steady_clock::now() - t_induce).count();
        if (rc) return fail(ctx_, rc, "restricting the source trees");
        for (size_t j = 0; j < jobs.size(); ++j) {
            Child &child = pending[j].res->children[pending[j].child];
            child.forest = jobs[j].out;
            // taxa of the component that are a tip of some kept tree; the others are attached as singleton
            // children (ref: scs.py:168-171).  A child left without trees raises when its wave is processed.
            const bool empty = scs_forest_num_trees(child.forest) == 0;
            for (int32_t x : pending[j].members) {
                if (present_[x]) child.taxa.push_back(x);
                else if (!empty) child.missing.push_back(x);
                present_[x] = 0;
            }
        }
        return SCS_OK;
    }

    // ref: scs.py:139-174 -- attach the children to the output tree and queue the sub-problems
    void emit(Task &task, SplitResult &res, std::vector<Task> &next) {
        if (!partitioned_ && !cooperative_) out_.shared_records += 1;
        if (record_) {
            scs_supertree::Record rec;
            rec.taxa = task.taxa;
            rec.part = res.part;
            rec.stats = res.stats;
            rec.wave = static_cast<int32_t>(out_.waves - 1);
            (task.shared ? sh_records_ : out_.records).push_back(std::move(rec));
        }
        for (Child &child : res.children) {
            // the children of a shared node are shared nodes: every rank creates them, in the same order
            const int32_t slot = add(task.slot, -1, task.shared);
            if (child.kind == CHILD_DEALT_AWAY) continue;
            if (!child.forest) {
                fill_star(slot, child.star.data(), static_cast<int>(child.star.size()), task.shared);
                continue;
            }
            const bool stays = child.kind == CHILD_SHARED;
            (child.kind == CHILD_DEALT_HERE ? backlog_ : next)
                .push_back(Task{child.forest, true, slot, std::move(child.taxa), stays});
            child.forest = nullptr;
            // taxa in no restricted tree (scs.py:168-171): known to whoever restricted, i.e. to every rank only
            // if the child stays shared
            for (int32_t x : child.missing) add(task.slot, x, task.shared && stays);
        }
    }

    scs_ctx *ctx_;
    int weighting_, contract_;
    uint64_t seed_;
    bool record_;
    int rank_ = 0, world_ = 1;
    bool partitioned_ = false;
    bool cooperative_ = false;
    std::vector<double> load_;                         // cooperative build: estimated work dealt to each rank
    std::vector<Task> backlog_;                        // ... and the sub-problems dealt to this rank
    std::vector<int32_t> sh_parent_, sh_taxon_;        // ... the shared node list
    std::vector<scs_supertree::Record> sh_records_;    // ... records of the shared nodes
    const bool trace_ = std::getenv("SCS_DRIVER_TRACE") != nullptr;
    double trace_induce_ = 0.0, trace_present_ = 0.0;  // thread-seconds (summed over host threads)
    scs_supertree &out_;
    int num_taxa_ = 0;
    std::vector<Scratch> scratch_, scratch_small_, scratch_medium_;
    scs_ctx *small_ctx_ = nullptr, *medium_ctx_ = nullptr;
    std::vector<TourBuffers> medium_buffers_;
    double medium_seconds_ = 0.0, medium_tour_seconds_ = 0.0;  // written by the thread that runs the medium batch
    std::vector<int32_t> owner_;    // global taxon id -> restriction job of the current wave
    std::vector<uint8_t> present_;  // scratch of plan_wave (all zero between waves)
    std::vector<TourBuffers> buffers_;
    std::vector<int32_t> part_;
};

}  // namespace

}  // namespace scs

using namespace scs;

extern "C" {

int scs_nodes_split_small_host(scs_ctx *ctx, int num_nodes, const scs_small_node *nodes, int64_t L_total,
                               int64_t T_total, const int64_t *leaf_offsets, const int32_t *leaf_taxon,
                               const int32_t *adj_depth, const double *adj_val, const int32_t *root_depth,
                               const double *tree_weight, int contract_edges, int32_t *part, scs_node_stats *stats) {
    if (!ctx || num_nodes < 0 || !nodes || !part || !stats || L_total < 0 || T_total < 0) return SCS_ERR_INVALID;
    if (num_nodes == 0) return SCS_OK;
    cudaSetDevice(ctx->device);
    SmallStage st;
    int rc = small_stage(ctx, num_nodes, L_total, T_total, &st);
    if (rc) return rc;
    const size_t nB = static_cast<size_t>(num_nodes), nL = static_cast<size_t>(L_total), nT = static_cast<size_t>(T_total);
    std::memcpy(st.nodes(), nodes, nB * sizeof(scs_small_node));
    std::memcpy(st.off(), leaf_offsets, (nT + nB) * sizeof(int64_t));
    if (nL) {
        std::memcpy(st.val(), adj_val, nL * sizeof(double));
        std::memcpy(st.tax(), leaf_taxon, nL * sizeof(int32_t));
        std::memcpy(st.dep(), adj_depth, nL * sizeof(int32_t));
    }
    if (nT) {
        std::memcpy(st.w(), tree_weight, nT * sizeof(double));
        std::memcpy(st.root(), root_depth, nT * sizeof(int32_t));
    }
    return small_run(ctx, num_nodes, st, contract_edges, part, stats);
}

int scs_nodes_split_small_dev(scs_ctx *ctx, int num_nodes, const scs_small_node *nodes_dev,
                              const int64_t *leaf_offsets_dev, const int32_t *leaf_taxon_dev,
                              const int32_t *adj_depth_dev, const double *adj_val_dev, const int32_t *root_depth_dev,
                              const double *tree_weight_dev, int contract_edges, int32_t *part_dev,
                              scs_node_stats *stats_dev) {
    if (!ctx || num_nodes < 0 || !nodes_dev || !part_dev || !stats_dev) return SCS_ERR_INVALID;
    cudaSetDevice(ctx->device);
    int32_t *bad_dev;
    int rc;
    if ((rc = reserve_as(ctx, SLOT_SCALARS, 64, &bad_dev))) return rc;
    return small_batch(ctx, num_nodes, nodes_dev, leaf_offsets_dev, leaf_taxon_dev, adj_depth_dev, adj_val_dev,
                       root_depth_dev, tree_weight_dev, contract_edges, part_dev, stats_dev, bad_dev);
}

int scs_supertree_build_sharded(scs_ctx *ctx, const scs_forest *forest, int weighting, int contract_edges,
                                uint64_t seed, int record_nodes, int rank, int world, scs_supertree **out) {
    if (!ctx || !forest || !out || weighting < 0 || weighting > 3 || world < 1 || rank < 0 || rank >= world)
        return SCS_ERR_INVALID;
    *out = nullptr;
    cudaSetDevice(ctx->device);
    std::unique_ptr<scs_supertree> result(new scs_supertree());
    int rc;
    const ShardState &sh = ctx->shard;
    const bool cooperative = world > 1 && sh.connected && sh.world == world && sh.rank == rank;
    if (ctx->device_forest && (world == 1 || cooperative)) {
        // the source trees go to the device once and stay there for the whole recursion (devdriver.cu)
        const scs_device_forest *resident = nullptr;
        const auto t0 = std::chrono::steady_clock::now();
        if ((rc = device_forest_refresh(ctx, forest, weighting, cooperative, &resident))) return rc;
        const auto t1 = std::chrono::steady_clock::now();
        rc = run_device_driver(ctx, resident, contract_edges, seed, record_nodes != 0, rank, world, result.get());
        const auto t2 = std::chrono::steady_clock::now();
        if (std::getenv("SCS_DRIVER_TRACE")) {
            auto ms = [](auto a, auto b) { return 1e3 * std::chrono::duration<double>(b - a).count(); };
            std::fprintf(stderr, "[scs build] rank %d: forest to the device %.2f ms, recursion %.2f ms, release %.2f ms\n", rank,
                         ms(t0, t1), ms(t1, t2), ms(t2, std::chrono::steady_clock::now()));
        }
    } else {
        Driver driver(ctx, weighting, contract_edges, seed, record_nodes != 0, rank, world, result.get());
        rc = driver.run(forest);
    }
    if (rc) return rc;
    if (world > 1 && result->shared_prefix == 0) result->shared_prefix = static_cast<int64_t>(result->parent.size());
    *out = result.release();
    return SCS_OK;
}

int scs_supertree_build_resident(scs_ctx *ctx, const scs_device_forest *forest, int contract_edges, uint64_t seed,
                                 int record_nodes, int rank, int world, scs_supertree **out) {
    if (!ctx || !forest || !out || world < 1 || rank < 0 || rank >= world) return SCS_ERR_INVALID;
    *out = nullptr;
    cudaSetDevice(ctx->device);
    std::unique_ptr<scs_supertree> result(new scs_supertree());
    const int rc = run_device_driver(ctx, forest, contract_edges, seed, record_nodes != 0, rank, world, result.get());
    if (rc) return rc;
    if (world > 1 && result->shared_prefix == 0) result->shared_prefix = static_cast<int64_t>(result->parent.size());
    *out = result.release();
    return SCS_OK;
}

int scs_supertree_build(scs_ctx *ctx, const scs_forest *forest, int weighting, int contract_edges, uint64_t seed,
                        int record_nodes, scs_supertree **out) {
    return scs_supertree_build_sharded(ctx, forest, weighting, contract_edges, seed, record_nodes, 0, 1, out);
}

int64_t scs_supertree_shared_prefix(const scs_supertree *tree) { return tree ? tree->shared_prefix : 0; }

int64_t scs_supertree_shared_records(const scs_supertree *tree) { return tree ? tree->shared_records : 0; }

int scs_supertree_wave_seconds(const scs_supertree *tree, double *seconds3) {
    if (!tree || !seconds3) return SCS_ERR_INVALID;
    std::memcpy(seconds3, tree->wave_seconds.data(), sizeof(double) * tree->wave_seconds.size());
    return static_cast<int>(tree->wave_seconds.size() / 3);
}

int scs_supertree_wave_info(const scs_supertree *tree, int32_t *tasks, int32_t *max_n) {
    if (!tree) return SCS_ERR_INVALID;
    const size_t count = tree->wave_tasks.size();
    if (tasks) std::memcpy(tasks, tree->wave_tasks.data(), sizeof(int32_t) * count);
    if (max_n) std::memcpy(max_n, tree->wave_max_n.data(), sizeof(int32_t) * count);
    return static_cast<int>(count);
}

int scs_supertree_destroy(scs_supertree *tree) {
    delete tree;
    return SCS_OK;
}

int64_t scs_supertree_num_nodes(const scs_supertree *tree) { return tree ? static_cast<int64_t>(tree->parent.size()) : 0; }

int scs_supertree_nodes(const scs_supertree *tree, int32_t *parent, int32_t *taxon) {
    if (!tree || !parent || !taxon) return SCS_ERR_INVALID;
    std::memcpy(parent, tree->parent.data(), sizeof(int32_t) * tree->parent.size());
    std::memcpy(taxon, tree->taxon.data(), sizeof(int32_t) * tree->taxon.size());
    return SCS_OK;
}

int scs_supertree_seconds(const scs_supertree *tree, double *seconds4) {
    if (!tree || !seconds4) return SCS_ERR_INVALID;
    for (int i = 0; i < 4; ++i) seconds4[i] = tree->seconds[i];
    return SCS_OK;
}

int scs_supertree_counters(const scs_supertree *tree, int64_t *nodes_small, int64_t *nodes_large, int64_t *waves,
                           int64_t *pair_visits) {
    if (!tree) return SCS_ERR_INVALID;
    if (nodes_small) *nodes_small = tree->nodes_small;
    if (nodes_large) *nodes_large = tree->nodes_large;
    if (waves) *waves = tree->waves;
    if (pair_visits) *pair_visits = tree->pair_visits;
    return SCS_OK;
}

int scs_supertree_medium_info(const scs_supertree *tree, int64_t *nodes_medium, int64_t *nodes_rerun, double *seconds) {
    if (!tree) return SCS_ERR_INVALID;
    if (nodes_medium) *nodes_medium = tree->nodes_medium;
    if (nodes_rerun) *nodes_rerun = tree->nodes_rerun;
    if (seconds) *seconds = tree->medium_seconds;
    return SCS_OK;
}

int64_t scs_supertree_num_records(const scs_supertree *tree) {
    return tree ? static_cast<int64_t>(tree->records.size()) : 0;
}

int scs_supertree_record_size(const scs_supertree *tree, int64_t index) {
    if (!tree || index < 0 || index >= static_cast<int64_t>(tree->records.size())) return SCS_ERR_INVALID;
    return static_cast<int>(tree->records[index].taxa.size());
}

int scs_supertree_record_wave(const scs_supertree *tree, int64_t index) {
    if (!tree || index < 0 || index >= static_cast<int64_t>(tree->records.size())) return SCS_ERR_INVALID;
    return tree->records[index].wave;
}

int scs_nodes_split_medium_dev(scs_ctx *ctx, int num_nodes, const int32_t *node_n, const int32_t *tree_begin,
                               const int64_t *part_offset, const uint64_t *seeds, int T, int64_t L,
                               const int64_t *leaf_offsets_dev, const int32_t *leaf_taxon_dev, const int32_t *adj_depth_dev,
                               const double *adj_val_dev, const int32_t *root_depth_dev, const double *tree_weight_dev,
                               int contract_edges, int32_t *part_dev, scs_node_stats *stats, uint8_t *needs_rerun) {
    if (!ctx) return SCS_ERR_INVALID;
    cudaSetDevice(ctx->device);
    return medium_batch(ctx, num_nodes, node_n, tree_begin, tree_begin + 1, part_offset, seeds, T, L, leaf_offsets_dev, leaf_taxon_dev,
                        adj_depth_dev, adj_val_dev, root_depth_dev, tree_weight_dev, contract_edges, part_dev, stats,
                        needs_rerun);
}

int scs_supertree_record(const scs_supertree *tree, int64_t index, int32_t *taxa, int32_t *part, scs_node_stats *stats) {
    if (!tree || index < 0 || index >= static_cast<int64_t>(tree->records.size())) return SCS_ERR_INVALID;
    const scs_supertree::Record &rec = tree->records[index];
    if (taxa) std::memcpy(taxa, rec.taxa.data(), sizeof(int32_t) * rec.taxa.size());
    if (part) std::memcpy(part, rec.part.data(), sizeof(int32_t) * rec.part.size());
    if (stats) *stats = rec.stats;
    return SCS_OK;
}

}  // extern "C"
