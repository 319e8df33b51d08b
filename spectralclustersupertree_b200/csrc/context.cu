// Context, workspace and the exported C ABI of libscs_b200.so (declared in include/scs_b200.h).
//
// The reference has no FFI; the seam is the per-recursion-node block of its construct_supertree
// (/root/reference/src/sc_supertree/scs.py:110-134).  scs_node_split_host is that block for a
// caller holding host buffers; the *_dev entry points are its stages for a caller that keeps
// its data on the GPU.

#include "common.cuh"

#include <chrono>
#include <cmath>

#include <cuda_profiler_api.h>

namespace scs {

int fail(scs_ctx *ctx, int status, const char *what, cudaError_t err) {
    if (ctx) {
        ctx->last_error = what ? what : "";
        if (err != cudaSuccess) {
            ctx->last_error += ": ";
            ctx->last_error += cudaGetErrorString(err);
        }
    }
    return status;
}

int reserve(scs_ctx *ctx, Slot slot, size_t bytes, void **out) {
    DeviceBuffer &buf = ctx->slots[slot];
    if (bytes == 0) bytes = 16;
    if (buf.bytes < bytes) {
        // Stream-ordered allocation: growing a slot neither synchronises the device (cudaFree would)
        // nor stalls the other contexts working on this GPU; the old block is released in stream
        // order, after the work already queued on it.  Recursion nodes shrink, so the first (largest)
        // node sizes everything; the pool keeps released blocks for the next growth.
        const size_t want = bytes + bytes / 4 + 256;
        if (buf.ptr) {
            SCS_CUDA(ctx, cudaFreeAsync(buf.ptr, ctx->stream));
            buf.ptr = nullptr;
            buf.bytes = 0;
        }
        cudaError_t err = cudaMallocAsync(&buf.ptr, want, ctx->stream);
        if (err != cudaSuccess) {
            buf.ptr = nullptr;
            return fail(ctx, SCS_ERR_CUDA, "cudaMallocAsync (workspace)", err);
        }
        buf.bytes = want;
    }
    *out = buf.ptr;
    return SCS_OK;
}

int reserve_pinned(scs_ctx *ctx, size_t bytes, void **out) {
    if (ctx->pinned_bytes < bytes) {
        if (ctx->pinned) {
            SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            SCS_CUDA(ctx, cudaFreeHost(ctx->pinned));
            ctx->pinned = nullptr;
            ctx->pinned_bytes = 0;
        }
        size_t want = bytes < 4096 ? 4096 : 2 * bytes;
        SCS_CUDA(ctx, cudaMallocHost(&ctx->pinned, want));
        ctx->pinned_bytes = want;
    }
    *out = ctx->pinned;
    return SCS_OK;
}

int ensure_workers(scs_ctx *ctx, int count) {
    while (static_cast<int>(ctx->workers.size()) < count - 1) {
        scs_ctx *worker = nullptr;
        const int rc = scs_ctx_create(ctx->device, nullptr, &worker);
        if (rc) return fail(ctx, rc, "creating a worker context");
        worker->small_limit = ctx->small_limit;
        ctx->workers.push_back(worker);
    }
    for (scs_ctx *worker : ctx->workers) {
        worker->small_limit = ctx->small_limit;
        worker->full_rows = ctx->full_rows;
        worker->wide_entries = ctx->wide_entries;
    }
    return SCS_OK;
}

void profile_begin(scs_ctx *ctx, int kind, double bytes, double units) {
    if (!ctx->profile_on) return;
    scs_ctx::ProfileRecord rec;
    rec.kind = kind;
    rec.bytes = bytes;
    rec.units = units;
    if (cudaEventCreate(&rec.start) != cudaSuccess || cudaEventCreate(&rec.stop) != cudaSuccess) return;
    cudaEventRecord(rec.start, ctx->stream);
    ctx->profile.push_back(rec);
}

void profile_end(scs_ctx *ctx) {
    if (!ctx->profile_on || ctx->profile.empty()) return;
    cudaEventRecord(ctx->profile.back().stop, ctx->stream);
}

namespace {

struct DeviceGuard {
    int previous = -1;
    explicit DeviceGuard(int device) {
        cudaGetDevice(&previous);
        if (previous != device) cudaSetDevice(device);
    }
};

template <typename T>
int upload(scs_ctx *ctx, Slot slot, const T *host, size_t count, T **dev) {
    int rc = reserve_as(ctx, slot, count + 1, dev);
    if (rc) return rc;
    if (count) SCS_CUDA(ctx, cudaMemcpyAsync(*dev, host, count * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
    return SCS_OK;
}

__global__ void relabel_components(int n, const int32_t *__restrict__ label, const int32_t *__restrict__ rank,
                                   int32_t *__restrict__ part) {
    int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v < n) part[v] = rank[label[v]];
}

__global__ void mark_roots(int n, const int32_t *__restrict__ label, int32_t *__restrict__ flag) {
    int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v < n) flag[v] = label[v] == v;
}

__global__ void expand_sides(int n, const int32_t *__restrict__ group, const int32_t *__restrict__ side,
                             int32_t *__restrict__ part) {
    int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v < n) part[v] = side[group ? group[v] : v];
}

void clear_stats(scs_node_stats *s) {
    std::memset(s, 0, sizeof(*s));
    s->eig[0] = 0.0;
    s->eig[1] = s->eig[2] = std::nan("");
    s->residual = std::nan("");
    s->margin = std::nan("");
}

}  // namespace

// One recursion node on device-resident tours; part_dev[n] receives component index or side.
int node_split(scs_ctx *ctx, int n, int T, int64_t L, const int64_t *leaf_offsets, const int32_t *leaf_taxon,
               const int32_t *adj_depth, const double *adj_val, const int32_t *root_depth,
               const double *tree_weight, int contract_edges, uint64_t seed, int32_t *part_dev,
               int32_t *part_host, scs_node_stats *stats, bool tour_components) {
    auto number_components = [&](const int32_t *label) -> int {
        // number the components by smallest member (scs.py:139 iterates them in arbitrary order)
        int32_t *flag, *rank;
        int rc;
        if ((rc = reserve_as(ctx, SLOT_GROUP_PTR, 4 * static_cast<size_t>(n) + 8, &flag))) return rc;
        rank = flag + n;
        const int blocks = ceil_div(n, 256);
        mark_roots<<<blocks, 256, 0, ctx->stream>>>(n, label, flag);
        SCS_LAUNCHED(ctx, "mark_roots");
        if ((rc = exclusive_scan(ctx, n, flag, rank))) return rc;
        relabel_components<<<blocks, 256, 0, ctx->stream>>>(n, label, rank, part_dev);
        SCS_LAUNCHED(ctx, "relabel_components");
        if (part_host) {
            SCS_CUDA(ctx, cudaMemcpyAsync(part_host, part_dev, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, ctx->stream));
            ctx->d2h_bytes += static_cast<int64_t>(sizeof(int32_t)) * n;
            SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        }
        return SCS_OK;
    };
    if (tour_components && n > ctx->small_limit) {
        // A disconnected node needs no graph: its components come from the tours, one pass over the leaves.
        // Every rank of a sharded build sees the same tours, so all of them leave here together.
        const auto t0 = std::chrono::steady_clock::now();
        int32_t *label, *scalars;
        void *pin_v;
        int rc;
        if ((rc = reserve_as(ctx, SLOT_LABEL, static_cast<size_t>(n), &label))) return rc;
        if ((rc = reserve_as(ctx, SLOT_SCALARS, 64, &scalars))) return rc;
        if ((rc = reserve_pinned(ctx, 512, &pin_v))) return rc;
        SCS_CUDA(ctx, cudaMemsetAsync(scalars, 0, 16 * sizeof(int32_t), ctx->stream));
        if ((rc = tour_components_async(ctx, n, T, L, leaf_offsets, leaf_taxon, adj_depth, root_depth, label,
                                        scalars + 8, scalars)))
            return rc;
        int32_t *host_scalars = reinterpret_cast<int32_t *>(static_cast<unsigned char *>(pin_v) + 256);
        SCS_CUDA(ctx, cudaMemcpyAsync(host_scalars, scalars, 16 * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        ctx->stage_seconds[6] += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        if (host_scalars[0] != 0) return fail(ctx, SCS_ERR_INPUT, "leaf tour: taxon id out of range");
        if (host_scalars[8] != 1) {
            stats->n_components = host_scalars[8];
            stats->contracted_size = n;
            return number_components(label);
        }
    }
    if (shard_applies(ctx, n))
        return node_split_sharded(ctx, n, T, L, leaf_offsets, leaf_taxon, adj_depth, adj_val, root_depth, tree_weight,
                                  contract_edges, seed, part_dev, part_host, stats);
    const int words = scs_bit_words(n);
    const size_t nn = static_cast<size_t>(n) * n;
    double *W, *Wc, *degree, *degree_c;
    int32_t *occ, *label, *group, *side, *scalars;
    uint32_t *adj_bits, *max_bits;
    int rc;
    if ((rc = reserve_as(ctx, SLOT_W, nn, &W))) return rc;
    if ((rc = reserve_as(ctx, SLOT_OCC, static_cast<size_t>(n), &occ))) return rc;
    if ((rc = reserve_as(ctx, SLOT_ADJ_BITS, static_cast<size_t>(n) * words, &adj_bits))) return rc;
    if ((rc = reserve_as(ctx, SLOT_MAX_BITS, static_cast<size_t>(n) * words, &max_bits))) return rc;
    if ((rc = reserve_as(ctx, SLOT_DEGREE, static_cast<size_t>(n), &degree))) return rc;
    if ((rc = reserve_as(ctx, SLOT_LABEL, static_cast<size_t>(n), &label))) return rc;
    if ((rc = reserve_as(ctx, SLOT_SCALARS, 64, &scalars))) return rc;
    ctx->last_n = n;
    ctx->last_m = 0;
    void *pin_v;
    if ((rc = reserve_pinned(ctx, 512, &pin_v))) return rc;
    unsigned char *pin = static_cast<unsigned char *>(pin_v);
    auto fetch_part = [&]() -> int {
        if (part_host) {
            SCS_CUDA(ctx, cudaMemcpyAsync(part_host, part_dev, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, ctx->stream));
            ctx->d2h_bytes += static_cast<int64_t>(sizeof(int32_t)) * n;
        }
        return SCS_OK;
    };

    auto now = [] { return std::chrono::steady_clock::now(); };
    auto lap = [&](int slot, std::chrono::steady_clock::time_point &since) {
        const auto t = now();
        ctx->stage_seconds[slot] += std::chrono::duration<double>(t - since).count();
        since = t;
    };
    auto mark = now();
    if ((rc = pcg_build(ctx, n, T, L, leaf_offsets, leaf_taxon, adj_depth, adj_val, root_depth, tree_weight, W,
                        nullptr, occ, adj_bits, contract_edges ? max_bits : nullptr, degree)))
        return rc;

    if (n <= ctx->small_limit) {
        // everything after the graph build in one launch; one round trip for the whole node
        scs_node_stats *stats_dev;
        if ((rc = reserve_as(ctx, SLOT_NODE_STATS, 1, &stats_dev))) return rc;
        if ((rc = reserve_as(ctx, SLOT_WC, nn, &Wc))) return rc;
        if ((rc = reserve_as(ctx, SLOT_GROUP, static_cast<size_t>(n), &group))) return rc;
        if ((rc = small_node(ctx, n, contract_edges, W, adj_bits, max_bits, part_dev, stats_dev, group, Wc))) return rc;
        SCS_CUDA(ctx, cudaMemcpyAsync(pin, stats_dev, sizeof(scs_node_stats), cudaMemcpyDeviceToHost, ctx->stream));
        SCS_CUDA(ctx, cudaMemcpyAsync(pin + 256, scalars, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
        if ((rc = fetch_part())) return rc;
        SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (*reinterpret_cast<int32_t *>(pin + 256) != 0)
            return fail(ctx, SCS_ERR_INPUT, "leaf tour: taxon id out of range");
        std::memcpy(stats, pin, sizeof(scs_node_stats));
        ctx->last_m = stats->contracted_size;
        if (stats->solver == -1) {
            stats->solver = 0;
            return fail(ctx, SCS_ERR_TOO_SMALL, "spectral step on a graph contracted to one vertex");
        }
        return SCS_OK;
    }

    // components of the graph and (speculatively) of the max-graph, then ONE round trip for: the
    // malformed-tour flag of the index kernel (scalars[0]), both component counts
    int32_t *label2 = nullptr;
    if ((rc = components_async(ctx, n, adj_bits, label, scalars + 8))) return rc;
    if (contract_edges) {
        if ((rc = reserve_as(ctx, SLOT_LABEL2, static_cast<size_t>(n), &label2))) return rc;
        if ((rc = components_async(ctx, n, max_bits, label2, scalars + 9))) return rc;
    }
    SCS_CUDA(ctx, cudaMemcpyAsync(pin + 256, scalars, 16 * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    lap(0, mark);  // enqueue of graph build + both component passes
    SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    lap(1, mark);  // their execution
    const int32_t *host_scalars = reinterpret_cast<const int32_t *>(pin + 256);
    if (host_scalars[0] != 0) return fail(ctx, SCS_ERR_INPUT, "leaf tour: taxon id out of range");
    const int ncomp = host_scalars[8];
    stats->n_components = ncomp;
    stats->contracted_size = n;
    const int blocks = ceil_div(n, 256);

    if (ncomp != 1) return number_components(label);

    int m = n;
    const double *Wm = W;
    const double *deg_m = degree;
    const int32_t *group_m = nullptr;
    if (contract_edges) {
        m = host_scalars[9];
        if ((rc = reserve_as(ctx, SLOT_WC, nn, &Wc))) return rc;
        if ((rc = reserve_as(ctx, SLOT_DEGREE_C, static_cast<size_t>(n), &degree_c))) return rc;
        if ((rc = reserve_as(ctx, SLOT_GROUP, static_cast<size_t>(n), &group))) return rc;
        if ((rc = contract_with_labels(ctx, n, W, adj_bits, label2, m, group, Wc, degree_c))) return rc;
        if (m != n) {
            Wm = Wc;
            deg_m = degree_c;
            group_m = group;
        }
    }
    ctx->last_m = m;
    stats->contracted_size = m;
    stats->spectral_ran = 1;
    if ((rc = reserve_as(ctx, SLOT_SIDE, static_cast<size_t>(n), &side))) return rc;
    if (m < 2) {
        // every taxon always sits with every other: the reference hands sklearn a 1 x 1 matrix and
        // it raises (ensure_min_samples=2, _spectral.py:699)
        return fail(ctx, SCS_ERR_TOO_SMALL, "spectral step on a graph contracted to one vertex");
    }
    lap(2, mark);  // enqueue of the contraction
    if ((rc = spectral_bipartition(ctx, m, Wm, deg_m, seed, side, stats))) return rc;
    lap(3, mark);  // spectral step (contraction execution included)
    expand_sides<<<blocks, 256, 0, ctx->stream>>>(n, group_m, side, part_dev);
    SCS_LAUNCHED(ctx, "expand_sides");
    if ((rc = fetch_part())) return rc;
    if (part_host) SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    lap(4, mark);  // result copy
    return SCS_OK;
}

}  // namespace scs

using namespace scs;

// Size the large buffers of a context for a node of n taxa, T trees, L leaves before it is used.  The driver
// calls this for every worker context with the largest node of a wave, so that which worker happens to draw
// which node (dynamic scheduling) never decides whether a timed run pays for a first allocation.
namespace scs {
int prewarm_node(scs_ctx *ctx, int n, int T, int64_t L) {
    DeviceGuard guard(ctx->device);
    const size_t nT = static_cast<size_t>(T), nL = static_cast<size_t>(L), nn = static_cast<size_t>(n) * n;
    const size_t total = (nT + 1) * sizeof(int64_t) + nL * (sizeof(double) + 2 * sizeof(int32_t)) +
                         nT * (sizeof(double) + sizeof(int32_t)) + 64;
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
    const size_t words = static_cast<size_t>(scs_bit_words(n));
    const size_t basis = static_cast<size_t>((n - 1 < 256 ? n - 1 : 256) + 3) * n;
    void *p;
    int rc;
    if ((rc = reserve(ctx, SLOT_TOUR_OFFSETS, total, &p))) return rc;
    if ((rc = reserve(ctx, SLOT_W, 8 * nn, &p))) return rc;
    if ((rc = reserve(ctx, SLOT_WC, 8 * nn, &p))) return rc;
    if ((rc = reserve(ctx, SLOT_ADJ_BITS, 4 * n * words, &p))) return rc;
    if ((rc = reserve(ctx, SLOT_MAX_BITS, 4 * n * words, &p))) return rc;
    if ((rc = reserve(ctx, SLOT_BASIS, 8 * basis, &p))) return rc;
    if ((rc = reserve(ctx, SLOT_LINKS, 16 * (nL + 1), &p))) return rc;
    if ((rc = reserve(ctx, SLOT_ENTRIES, 8 * (nL + 1), &p))) return rc;
    if ((rc = reserve(ctx, SLOT_BUCKET_COUNT, 448 * (nL + 1), &p))) return rc;  // LeafStairs (pcg.cu)
    if ((rc = reserve(ctx, SLOT_START16, 64 * (nL + 1), &p))) return rc;
    return SCS_OK;
}
}  // namespace scs

namespace scs {
int node_split_host(scs_ctx *ctx, int n, int T, int64_t L, const int64_t *leaf_offsets, const int32_t *leaf_taxon,
                    const int32_t *adj_depth, const double *adj_val, const int32_t *root_depth,
                    const double *tree_weight, int contract_edges, uint64_t seed, int32_t *part,
                    scs_node_stats *stats_out, bool tour_components) {
    if (!ctx) return SCS_ERR_INVALID;
    if (n <= 0 || T < 0 || L < 0 || !part) return fail(ctx, SCS_ERR_INVALID, "node_split: bad argument");
    if (T > 0 && (!leaf_offsets || !root_depth || !tree_weight))
        return fail(ctx, SCS_ERR_INVALID, "node_split: null tour array");
    if (L > 0 && (!leaf_taxon || !adj_depth || !adj_val))
        return fail(ctx, SCS_ERR_INVALID, "node_split: null tour array");
    DeviceGuard guard(ctx->device);
    scs_node_stats local;
    scs_node_stats *stats = stats_out ? stats_out : &local;
    clear_stats(stats);

    // stage the tours through one pinned buffer so the copies are truly asynchronous
    const size_t nT = static_cast<size_t>(T), nL = static_cast<size_t>(L);
    const size_t b_off = (nT + 1) * sizeof(int64_t);
    const size_t b_val = nL * sizeof(double);
    const size_t b_w = nT * sizeof(double);
    const size_t b_tax = nL * sizeof(int32_t);
    const size_t b_dep = nL * sizeof(int32_t);
    const size_t b_root = nT * sizeof(int32_t);
    const size_t total = b_off + b_val + b_w + b_tax + b_dep + b_root + 64;
    int rc;
    if (ctx->pinned_io_bytes < total) {
        if (ctx->pinned_io) {
            SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            SCS_CUDA(ctx, cudaFreeHost(ctx->pinned_io));
            ctx->pinned_io = nullptr;
            ctx->pinned_io_bytes = 0;
        }
        const size_t want = 2 * total + 4096;  // pinned allocations synchronise the device: grow rarely
        SCS_CUDA(ctx, cudaMallocHost(&ctx->pinned_io, want));
        ctx->pinned_io_bytes = want;
    }
    unsigned char *stage = static_cast<unsigned char *>(ctx->pinned_io);
    unsigned char *dev_stage;
    if ((rc = reserve_as(ctx, SLOT_TOUR_OFFSETS, total, &dev_stage))) return rc;
    size_t o_off = 0, o_val = o_off + b_off, o_w = o_val + b_val, o_tax = o_w + b_w, o_dep = o_tax + b_tax,
           o_root = o_dep + b_dep;
    if (T > 0) {
        std::memcpy(stage + o_off, leaf_offsets, b_off);
        std::memcpy(stage + o_w, tree_weight, b_w);
        std::memcpy(stage + o_root, root_depth, b_root);
    } else {
        std::memset(stage + o_off, 0, b_off);
    }
    if (L > 0) {
        std::memcpy(stage + o_val, adj_val, b_val);
        std::memcpy(stage + o_tax, leaf_taxon, b_tax);
        std::memcpy(stage + o_dep, adj_depth, b_dep);
    }
    SCS_CUDA(ctx, cudaMemcpyAsync(dev_stage, stage, total - 64, cudaMemcpyHostToDevice, ctx->stream));
    ctx->h2d_bytes += static_cast<int64_t>(total - 64);
    ctx->pending_units = 0.0;
    for (int t = 0; t < T; ++t) {
        const double k = static_cast<double>(leaf_offsets[t + 1] - leaf_offsets[t]);
        ctx->pending_units += k * (k - 1.0);
    }

    int32_t *part_dev;
    if ((rc = reserve_as(ctx, SLOT_PART, static_cast<size_t>(n), &part_dev))) return rc;
    rc = node_split(ctx, n, T, L, reinterpret_cast<const int64_t *>(dev_stage + o_off),
                    reinterpret_cast<const int32_t *>(dev_stage + o_tax),
                    reinterpret_cast<const int32_t *>(dev_stage + o_dep),
                    reinterpret_cast<const double *>(dev_stage + o_val),
                    reinterpret_cast<const int32_t *>(dev_stage + o_root),
                    reinterpret_cast<const double *>(dev_stage + o_w), contract_edges, seed, part_dev, part, stats,
                    tour_components);
    ctx->pending_units = 0.0;
    return rc;
}
}  // namespace scs

extern "C" {

int scs_version(void) { return 100; }

const char *scs_status_string(int status) {
    switch (status) {
    case SCS_OK: return "ok";
    case SCS_ERR_INVALID: return "invalid argument";
    case SCS_ERR_CUDA: return "CUDA error";
    case SCS_ERR_NO_DEVICE: return "no usable CUDA device";
    case SCS_ERR_TOO_SMALL: return "fewer than two vertices in the spectral step";
    case SCS_ERR_NO_CONVERGE: return "eigensolver did not converge";
    case SCS_ERR_INPUT: return "malformed input";
    case SCS_ERR_EMPTY: return "there must be at least one tree to make a supertree";
    case SCS_ERR_PEER: return "a wait for a peer GPU timed out";
    default: return "unknown status";
    }
}

const char *scs_last_error(const scs_ctx *ctx) { return ctx ? ctx->last_error.c_str() : ""; }

int scs_bit_words(int n) { return (n + 31) / 32; }

int scs_ctx_create(int device, void *stream, scs_ctx **out) {
    if (!out) return SCS_ERR_INVALID;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) {
        cudaGetLastError();
        return SCS_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= count) return SCS_ERR_INVALID;
    if (cudaSetDevice(device) != cudaSuccess) return SCS_ERR_CUDA;
    scs_ctx *ctx = new scs_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
        delete ctx;
        return SCS_ERR_CUDA;
    }
    {
        // never hand pooled workspace back to the driver between recursion nodes
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            uint64_t threshold = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &threshold);
        }
        cudaGetLastError();
    }
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    ctx->smem_per_sm = prop.sharedMemPerMultiprocessor;
    if (stream) {
        ctx->stream = static_cast<cudaStream_t>(stream);
    } else {
        if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
            delete ctx;
            return SCS_ERR_CUDA;
        }
        ctx->own_stream = true;
    }
    *out = ctx;
    return SCS_OK;
}

int scs_ctx_destroy(scs_ctx *ctx) {
    if (!ctx) return SCS_OK;
    DeviceGuard guard(ctx->device);
    for (scs_ctx *worker : ctx->workers) scs_ctx_destroy(worker);
    ctx->workers.clear();
    cudaStreamSynchronize(ctx->stream);
    if (ctx->driver_cache && ctx->driver_cache_release) ctx->driver_cache_release(ctx, ctx->driver_cache);
    ctx->driver_cache = nullptr;
    scs_shard_destroy(ctx);
    for (auto &buf : ctx->slots)
        if (buf.ptr) cudaFreeAsync(buf.ptr, ctx->stream);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    if (ctx->pinned_io) cudaFreeHost(ctx->pinned_io);
    for (auto &rec : ctx->profile) {
        cudaEventDestroy(rec.start);
        cudaEventDestroy(rec.stop);
    }
    if (ctx->timer_start) cudaEventDestroy(ctx->timer_start);
    if (ctx->timer_stop) cudaEventDestroy(ctx->timer_stop);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return SCS_OK;
}

int scs_ctx_synchronize(scs_ctx *ctx) {
    if (!ctx) return SCS_ERR_INVALID;
    DeviceGuard guard(ctx->device);
    SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SCS_OK;
}

int64_t scs_ctx_launch_count(const scs_ctx *ctx) { return ctx ? ctx->launches : 0; }

int scs_ctx_io_bytes(const scs_ctx *ctx, int64_t *h2d, int64_t *d2h) {
    if (!ctx) return SCS_ERR_INVALID;
    if (h2d) *h2d = ctx->h2d_bytes;
    if (d2h) *d2h = ctx->d2h_bytes;
    return SCS_OK;
}

int scs_ctx_timer_start(scs_ctx *ctx) {
    if (!ctx) return SCS_ERR_INVALID;
    DeviceGuard guard(ctx->device);
    if (!ctx->timer_start) {
        SCS_CUDA(ctx, cudaEventCreate(&ctx->timer_start));
        SCS_CUDA(ctx, cudaEventCreate(&ctx->timer_stop));
    }
    SCS_CUDA(ctx, cudaEventRecord(ctx->timer_start, ctx->stream));
    return SCS_OK;
}

int scs_ctx_timer_stop(scs_ctx *ctx, double *ms) {
    if (!ctx || !ms || !ctx->timer_start) return SCS_ERR_INVALID;
    DeviceGuard guard(ctx->device);
    SCS_CUDA(ctx, cudaEventRecord(ctx->timer_stop, ctx->stream));
    SCS_CUDA(ctx, cudaEventSynchronize(ctx->timer_stop));
    float t = 0.0f;
    SCS_CUDA(ctx, cudaEventElapsedTime(&t, ctx->timer_start, ctx->timer_stop));
    *ms = t;
    return SCS_OK;
}

int scs_ctx_set_small_node_limit(scs_ctx *ctx, int limit) {
    if (!ctx || limit < 0) return SCS_ERR_INVALID;
    ctx->small_limit = limit > kSmallNode ? kSmallNode : limit;
    return SCS_OK;
}

int scs_ctx_set_medium_node_limit(scs_ctx *ctx, int limit) {
    if (!ctx || limit < 0) return SCS_ERR_INVALID;
    ctx->medium_limit = limit > kMediumMax ? kMediumMax : limit;
    return SCS_OK;
}

int scs_ctx_set_device_forest(scs_ctx *ctx, int on) {
    if (!ctx) return SCS_ERR_INVALID;
    ctx->device_forest = on != 0;
    return SCS_OK;
}

int scs_ctx_set_wide_entries(scs_ctx *ctx, int on) {
    if (!ctx) return SCS_ERR_INVALID;
    ctx->wide_entries = on != 0;
    return SCS_OK;
}

int scs_ctx_set_full_rows(scs_ctx *ctx, int on) {
    if (!ctx) return SCS_ERR_INVALID;
    ctx->full_rows = on != 0;
    for (scs_ctx *worker : ctx->workers) worker->full_rows = ctx->full_rows;
    return SCS_OK;
}

int scs_ctx_stage_seconds(scs_ctx *ctx, double *seconds8, int reset) {
    if (!ctx || !seconds8) return SCS_ERR_INVALID;
    for (int i = 0; i < 8; ++i) {
        seconds8[i] = ctx->stage_seconds[i];
        if (reset) ctx->stage_seconds[i] = 0.0;
    }
    return SCS_OK;
}

int scs_ctx_flush_l2(scs_ctx *ctx) {
    if (!ctx) return SCS_ERR_INVALID;
    DeviceGuard guard(ctx->device);
    const size_t bytes = 256u << 20;  // twice the 126 MB L2
    void *buf;
    int rc = reserve(ctx, SLOT_L2_FLUSH, bytes, &buf);
    if (rc) return rc;
    ctx->flush_value += 1;
    SCS_CUDA(ctx, cudaMemsetAsync(buf, ctx->flush_value & 0xff, bytes, ctx->stream));
    SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SCS_OK;
}

int scs_ctx_profile_enable(scs_ctx *ctx, int on) {
    if (!ctx) return SCS_ERR_INVALID;
    ctx->profile_on = on != 0;
    return SCS_OK;
}

int scs_ctx_profile_read(scs_ctx *ctx, int kind, int64_t *launches, double *ms, double *bytes, double *units) {
    if (!ctx || kind < 0 || kind >= PROFILE_KINDS) return SCS_ERR_INVALID;
    DeviceGuard guard(ctx->device);
    SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    int64_t count = 0;
    double total_ms = 0.0, total_bytes = 0.0, total_units = 0.0;
    std::vector<scs_ctx::ProfileRecord> keep;
    for (auto &rec : ctx->profile) {
        if (rec.kind != kind) {
            keep.push_back(rec);
            continue;
        }
        float t = 0.0f;
        if (cudaEventElapsedTime(&t, rec.start, rec.stop) == cudaSuccess) {
            count += 1;
            total_ms += t;
            total_bytes += rec.bytes;
            total_units += rec.units;
        }
        cudaEventDestroy(rec.start);
        cudaEventDestroy(rec.stop);
    }
    cudaGetLastError();
    ctx->profile.swap(keep);
    if (launches) *launches = count;
    if (ms) *ms = total_ms;
    if (bytes) *bytes = total_bytes;
    if (units) *units = total_units;
    return SCS_OK;
}

int scs_debug_small_cycles(scs_ctx *ctx, uint64_t *cycles2, int reset) {
    if (!ctx || !cycles2) return SCS_ERR_INVALID;
    DeviceGuard guard(ctx->device);
    unsigned long long raw[2] = {0, 0};
    const int rc = small_cycles(ctx, raw, reset);
    cycles2[0] = raw[0];
    cycles2[1] = raw[1];
    return rc;
}

int scs_profiler_range(int on) {
    const cudaError_t err = on ? cudaProfilerStart() : cudaProfilerStop();
    return err == cudaSuccess ? SCS_OK : SCS_ERR_CUDA;
}

int scs_pcg_build_dev(scs_ctx *ctx, int n, int T, int64_t L, const int64_t *leaf_offsets_dev,
                      const int32_t *leaf_taxon_dev, const int32_t *adj_depth_dev, const double *adj_val_dev,
                      const int32_t *root_depth_dev, const double *tree_weight_dev, double *W_dev, int32_t *C_dev,
                      int32_t *occ_dev, uint32_t *adj_bits_dev, uint32_t *max_bits_dev, double *degree_dev) {
    if (!ctx) return SCS_ERR_INVALID;
    DeviceGuard guard(ctx->device);
    return pcg_build(ctx, n, T, L, leaf_offsets_dev, leaf_taxon_dev, adj_depth_dev, adj_val_dev, root_depth_dev,
                     tree_weight_dev, W_dev, C_dev, occ_dev, adj_bits_dev, max_bits_dev, degree_dev);
}

int scs_pcg_build_rows_dev(scs_ctx *ctx, int n, int T, int64_t L, const int64_t *leaf_offsets_dev,
                           const int32_t *leaf_taxon_dev, const int32_t *adj_depth_dev, const double *adj_val_dev,
                           const int32_t *root_depth_dev, const double *tree_weight_dev, int row0, int row1,
                           double *W_rows_dev, int32_t *occ_dev, uint32_t *adj_bits_dev, uint32_t *max_bits_dev,
                           double *degree_dev) {
    if (!ctx) return SCS_ERR_INVALID;
    DeviceGuard guard(ctx->device);
    RowBlock rows;
    rows.row0 = row0;
    rows.row1 = row1;
    return pcg_build(ctx, n, T, L, leaf_offsets_dev, leaf_taxon_dev, adj_depth_dev, adj_val_dev, root_depth_dev,
                     tree_weight_dev, W_rows_dev, nullptr, occ_dev, adj_bits_dev, max_bits_dev, degree_dev, rows);
}

int scs_components_dev(scs_ctx *ctx, int n, const uint32_t *bits_dev, int32_t *label_dev,
                       int32_t *n_components_host) {
    if (!ctx) return SCS_ERR_INVALID;
    DeviceGuard guard(ctx->device);
    return components(ctx, n, bits_dev, label_dev, n_components_host);
}

int scs_contract_dev(scs_ctx *ctx, int n, const double *W_dev, const uint32_t *adj_bits_dev,
                     const uint32_t *max_bits_dev, int32_t *group_dev, int32_t *m_host, double *Wc_dev,
                     double *degree_c_dev) {
    if (!ctx) return SCS_ERR_INVALID;
    DeviceGuard guard(ctx->device);
    return contract(ctx, n, W_dev, adj_bits_dev, max_bits_dev, group_dev, m_host, Wc_dev, degree_c_dev);
}

int scs_spectral_bipartition_dev(scs_ctx *ctx, int m, const double *W_dev, const double *degree_dev,
                                 uint64_t seed, int32_t *side_dev, scs_node_stats *stats_host) {
    if (!ctx) return SCS_ERR_INVALID;
    DeviceGuard guard(ctx->device);
    scs_node_stats local;
    scs_node_stats *stats = stats_host ? stats_host : &local;
    clear_stats(stats);
    stats->n_components = 1;
    stats->contracted_size = m;
    stats->spectral_ran = 1;
    if (m < 2) return fail(ctx, SCS_ERR_TOO_SMALL, "spectral step needs at least two vertices");
    return spectral_bipartition(ctx, m, W_dev, degree_dev, seed, side_dev, stats);
}

int scs_normalized_matvec_dev(scs_ctx *ctx, int m, const double *W_dev, const double *inv_sqrt_deg_dev,
                              const double *x_dev, double *y_dev) {
    if (!ctx) return SCS_ERR_INVALID;
    DeviceGuard guard(ctx->device);
    return normalized_matvec(ctx, m, W_dev, inv_sqrt_deg_dev, x_dev, y_dev);
}

int scs_node_split_dev(scs_ctx *ctx, int n, int T, int64_t L, const int64_t *leaf_offsets_dev,
                       const int32_t *leaf_taxon_dev, const int32_t *adj_depth_dev, const double *adj_val_dev,
                       const int32_t *root_depth_dev, const double *tree_weight_dev, int contract_edges,
                       uint64_t seed, int32_t *part_dev, scs_node_stats *stats_host) {
    if (!ctx || n <= 0 || !part_dev) return SCS_ERR_INVALID;
    DeviceGuard guard(ctx->device);
    scs_node_stats local;
    scs_node_stats *stats = stats_host ? stats_host : &local;
    clear_stats(stats);
    return node_split(ctx, n, T, L, leaf_offsets_dev, leaf_taxon_dev, adj_depth_dev, adj_val_dev, root_depth_dev,
                      tree_weight_dev, contract_edges, seed, part_dev, nullptr, stats);
}

int scs_node_split_host(scs_ctx *ctx, int n, int T, int64_t L, const int64_t *leaf_offsets,
                        const int32_t *leaf_taxon, const int32_t *adj_depth, const double *adj_val,
                        const int32_t *root_depth, const double *tree_weight, int contract_edges, uint64_t seed,
                        int32_t *part, scs_node_stats *stats_out) {
    return node_split_host(ctx, n, T, L, leaf_offsets, leaf_taxon, adj_depth, adj_val, root_depth, tree_weight,
                           contract_edges, seed, part, stats_out, false);
}

int scs_node_last_buffers(scs_ctx *ctx, int *n, int *m, double **W_dev, uint32_t **adj_bits_dev,
                          uint32_t **max_bits_dev, int32_t **occ_dev, double **degree_dev, double **Wc_dev,
                          int32_t **group_dev) {
    if (!ctx) return SCS_ERR_INVALID;
    if (n) *n = ctx->last_n;
    if (m) *m = ctx->last_m;
    if (W_dev) *W_dev = static_cast<double *>(ctx->slots[SLOT_W].ptr);
    if (adj_bits_dev) *adj_bits_dev = static_cast<uint32_t *>(ctx->slots[SLOT_ADJ_BITS].ptr);
    if (max_bits_dev) *max_bits_dev = static_cast<uint32_t *>(ctx->slots[SLOT_MAX_BITS].ptr);
    if (occ_dev) *occ_dev = static_cast<int32_t *>(ctx->slots[SLOT_OCC].ptr);
    if (degree_dev) *degree_dev = static_cast<double *>(ctx->slots[SLOT_DEGREE].ptr);
    if (Wc_dev) *Wc_dev = static_cast<double *>(ctx->slots[SLOT_WC].ptr);
    if (group_dev) *group_dev = static_cast<int32_t *>(ctx->slots[SLOT_GROUP].ptr);
    return SCS_OK;
}

int scs_memcpy_d2h(scs_ctx *ctx, void *host, const void *dev, size_t bytes) {
    if (!ctx || !host || !dev) return SCS_ERR_INVALID;
    DeviceGuard guard(ctx->device);
    SCS_CUDA(ctx, cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SCS_OK;
}

int scs_memcpy_h2d(scs_ctx *ctx, void *dev, const void *host, size_t bytes) {
    if (!ctx || !host || !dev) return SCS_ERR_INVALID;
    DeviceGuard guard(ctx->device);
    SCS_CUDA(ctx, cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SCS_OK;
}

int scs_dev_alloc(scs_ctx *ctx, size_t bytes, void **out) {
    if (!ctx || !out) return SCS_ERR_INVALID;
    DeviceGuard guard(ctx->device);
    SCS_CUDA(ctx, cudaMalloc(out, bytes ? bytes : 16));
    return SCS_OK;
}

int scs_dev_free(scs_ctx *ctx, void *ptr) {
    if (!ctx) return SCS_ERR_INVALID;
    DeviceGuard guard(ctx->device);
    SCS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    SCS_CUDA(ctx, cudaFree(ptr));
    return SCS_OK;
}

}  // extern "C"
