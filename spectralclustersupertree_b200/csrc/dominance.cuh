// The dominance-count row of the triplet passes (triplets.cu, pairwise.cu): a warp grows the window of restricted
// tour positions around a taxon a one depth level at a time, deepest first, and counts the taxa each level adds
// against those already inside with a Fenwick tree in shared memory.
#pragma once

#include "common.cuh"

namespace scs {

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

}  // namespace scs
