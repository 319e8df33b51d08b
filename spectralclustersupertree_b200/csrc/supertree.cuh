// Pieces shared by the passes that score a supertree against its source trees (support.cu, triplets.cu): the
// supertree in depth-first pre-order with the leaf range of every node, a CTA-wide exclusive scan and the rank of a
// leaf position in a bitmap.
#pragma once

#include <vector>

#include "common.cuh"

namespace scs {

// In-place exclusive prefix sum of data[0, n) by the whole CTA; returns the total.  sums: 33 shared ints.
__device__ inline int block_scan(int32_t *data, int n, int32_t *sums) {
    const int per = (n + blockDim.x - 1) / blockDim.x;
    const int b = min(n, static_cast<int>(threadIdx.x) * per), e = min(n, b + per);
    int own = 0;
    for (int i = b; i < e; ++i) own += data[i];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int inc = own;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int o = __shfl_up_sync(0xffffffffu, inc, off);
        if (lane >= off) inc += o;
    }
    if (lane == 31) sums[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const int v = lane < static_cast<int>(blockDim.x >> 5) ? sums[lane] : 0;
        int w = v;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const int o = __shfl_up_sync(0xffffffffu, w, off);
            if (lane >= off) w += o;
        }
        sums[lane] = w - v;
        if (lane == 31) sums[32] = w;
    }
    __syncthreads();
    int run = sums[warp] + inc - own;
    for (int i = b; i < e; ++i) {
        const int v = data[i];
        data[i] = run;
        run += v;
    }
    const int total = sums[32];
    __syncthreads();
    return total;
}

// Rank of bit p among the set bits of a bitmap, given the exclusive prefix of its word popcounts (wpre): how a tree's
// taxa get their order in S from a bitmap over S's leaf positions.
__device__ __forceinline__ int bitmap_rank(const uint32_t *bits, const int32_t *wpre, int p) {
    return wpre[p >> 5] + __popc(bits[p >> 5] & ((1u << (p & 31)) - 1u));
}

// The supertree in depth-first pre-order (children in index order) with the leaf range of every node.
struct PreorderTree {
    std::vector<int32_t> order, parent, first, count, pos;
    int32_t leaves = 0;
};

inline int preorder_supertree(int64_t num_nodes, const int32_t *parent, const int32_t *taxon, int taxa, PreorderTree *out) {
    if (parent[0] != -1) return SCS_ERR_INPUT;
    std::vector<int32_t> child_start(static_cast<size_t>(num_nodes) + 1, 0), child(static_cast<size_t>(num_nodes));
    for (int64_t i = 1; i < num_nodes; ++i) {
        if (parent[i] < 0 || parent[i] >= i) return SCS_ERR_INPUT;
        child_start[parent[i] + 1] += 1;
    }
    for (int64_t i = 0; i < num_nodes; ++i) child_start[i + 1] += child_start[i];
    {
        std::vector<int32_t> cursor(child_start.begin(), child_start.end() - 1);
        for (int64_t i = 1; i < num_nodes; ++i) child[cursor[parent[i]]++] = static_cast<int32_t>(i);
    }
    out->pos.assign(static_cast<size_t>(taxa > 0 ? taxa : 1), -1);
    std::vector<int32_t> pre_of(static_cast<size_t>(num_nodes));
    out->order.clear();
    out->order.reserve(static_cast<size_t>(num_nodes));
    out->parent.assign(static_cast<size_t>(num_nodes), -1);
    out->first.assign(static_cast<size_t>(num_nodes), 0);
    out->count.assign(static_cast<size_t>(num_nodes), 0);
    std::vector<int32_t> stack{0};
    int32_t leaves = 0;
    while (!stack.empty()) {
        const int32_t v = stack.back();
        stack.pop_back();
        const int32_t pre = static_cast<int32_t>(out->order.size());
        pre_of[v] = pre;
        out->order.push_back(v);
        out->parent[pre] = v == 0 ? -1 : pre_of[parent[v]];
        out->first[pre] = leaves;
        const bool tip = child_start[v + 1] == child_start[v];
        if (tip) {
            const int32_t x = taxon[v];
            if (x < 0 || x >= taxa || out->pos[x] >= 0) return SCS_ERR_INPUT;
            out->pos[x] = leaves++;
        } else {
            if (taxon[v] >= 0) return SCS_ERR_INPUT;
            for (int32_t c = child_start[v + 1] - 1; c >= child_start[v]; --c) stack.push_back(child[c]);
        }
    }
    for (int32_t u = static_cast<int32_t>(num_nodes) - 1; u >= 0; --u) {
        if (out->count[u] == 0) out->count[u] = 1;  // a tip (internal nodes have at least one leaf below)
        if (u > 0) out->count[out->parent[u]] += out->count[u];
    }
    out->leaves = leaves;
    return SCS_OK;
}

}  // namespace scs
