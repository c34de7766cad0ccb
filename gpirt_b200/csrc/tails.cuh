// Device helpers shared by the IRF bands (kernels.cu) and PSIS-LOO (loo.cu): log sigma of a linear predictor and the
// bounded per-cell heaps that keep one tail of a stream of draws.
#pragma once
#include "common.cuh"

namespace gpirt {

// sigma(a) and log sigma(a) from one exp and one log1p, both stable for either sign of a
__device__ __forceinline__ void log_sigmoid(double a, double& sig, double& ls) {
    const double e = exp(-fabs(a));
    sig = (a >= 0.0 ? 1.0 : e) / (1.0 + e);
    ls = -(fmax(-a, 0.0) + log1p(e));
}

// MAXH: max-heap (root = largest kept value); `above(a, b)`: a belongs nearer the root than b
template <bool MAXH>
__device__ __forceinline__ bool heap_above(double a, double b) { return MAXH ? a > b : a < b; }
// Adds v to the heap of cell c, stored slot-major (slot i at h[i * cells + c]), which holds `size` values (capacity K):
// while not full every value goes in (sift up); once full v replaces the root only if it belongs strictly below it in
// the kept tail (sift down).  Returns true when a value leaves the kept tail, in *out: v itself when it is rejected (ties
// keep the value already there), the old root when v evicts it.
template <bool MAXH>
__device__ __forceinline__ bool heap_add(double* h, int64_t cells, int64_t c, int K, int size, double v, double* out) {
    auto at = [&](int i) -> double& { return h[(int64_t)i * cells + c]; };
    if (size < K) {
        int i = size;
        while (i > 0) {
            const int p = (i - 1) >> 1;
            const double pv = at(p);
            if (!heap_above<MAXH>(v, pv)) break;
            at(i) = pv;
            i = p;
        }
        at(i) = v;
        return false;
    }
    const double root = at(0);
    if (!heap_above<MAXH>(root, v)) { *out = v; return true; }
    int i = 0;
    for (;;) {
        const int l = 2 * i + 1;
        if (l >= K) break;
        int ci = l;
        double cv = at(l);
        if (l + 1 < K) {
            const double rv = at(l + 1);
            if (heap_above<MAXH>(rv, cv)) { ci = l + 1; cv = rv; }
        }
        if (!heap_above<MAXH>(cv, v)) break;
        at(i) = cv;
        i = ci;
    }
    at(i) = v;
    *out = root;
    return true;
}

}  // namespace gpirt
