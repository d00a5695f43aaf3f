// dtfill_k4_exact.cuh -- K4x: evaluation.py:82-123, 196-239 with numpy's own summation order
#pragma once
#include <type_traits>

#include "dtfill_k4_metrics.cuh"

namespace dtfill {

// ------------------------------------------------------------------------------------------------------
// Result.evaluate / Result_NYU.evaluate take np.mean of four arrays of per-pixel terms over the valid pixels, compacted in
// raster order (output[valid_mask], evaluation.py:89-90 / :203-204).  np.mean is add.reduce in the arrays' dtype --
// float32 when the ground truth is float32 (eval_NYU.py), float64 when it is float64 (data_read.py:223) -- divided by the
// count in that dtype, and add.reduce over a contiguous array is numpy's pairwise summation:
//     n < 8:     0 + a[0] + a[1] + ...
//     n <= 128:  eight running sums r[j] += a[i + j] over the multiples of 8, ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)),
//                then the remaining n % 8 elements one by one
//     else:      n2 = n / 2 rounded down to a multiple of 8;  sum(a[0:n2]) + sum(a[n2:n])
// (numpy/_core/src/umath/loops_utils.h.src; pinned by tests/test_host_logic.py against np.add.reduce).  The kernels below
// reproduce exactly that tree, so the metrics are the reference's bit for bit -- the fixed-order float64 sums of
// k4_metrics_partial agree with numpy's float32 pairwise sums only to ~1e-5.
//   k4x_compact  one block per frame: the terms of the valid pixels, compacted in raster order (ballots + warp ranks);
//                the ground truth is stored as the arithmetic type or, in KITTI mode, as 16-bit PNG samples; the WIN
//                instance (NYU mode, float32) scores a crop window of the frames
//   k4x_reduce   one block per frame: the leaves (<= 128 elements) of the tree in parallel, then the tree itself
// Terms: 0 |d|^2, 1 |d| (KITTI) or |d| / t (NYU), 2 |dinv|^2, 3 |dinv|; counts: valid, delta1..3.
// ------------------------------------------------------------------------------------------------------
constexpr int K4X_THREADS = 1024;

// IEEE operations that the compiler may not contract into fused multiply-adds (numpy rounds every product)
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float sub_rn(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ double sub_rn(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ float sqrt_rn(float a) { return __fsqrt_rn(a); }
__device__ __forceinline__ double sqrt_rn(double a) { return __dsqrt_rn(a); }
__device__ __forceinline__ float div_rn(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ double div_rn(double a, double b) { return __ddiv_rn(a, b); }

template <typename GT, int MODE>
__device__ __forceinline__ bool metric_terms(float o, GT t, GT* term, int* hit)
{
    if (!((o > 0.01f) && (t > (GT)0.01))) return false;                // evaluation.py:85-87 / :199-201
    if (MODE == 0) {
        const GT o_mm = (GT)__fmul_rn(1e3f, o);                        // :89 float32 product
        const GT t_mm = mul_rn((GT)1e3, t);                            // :90
        const GT d = o_mm > t_mm ? sub_rn(o_mm, t_mm) : sub_rn(t_mm, o_mm);      // :92
        const GT io = (GT)__fdiv_rn(1.0f, __fmul_rn(1e-3f, o));        // :116
        const GT it = div_rn((GT)1.0, mul_rn((GT)1e-3, t));            // :117
        const GT di = io > it ? sub_rn(io, it) : sub_rn(it, io);       // :118
        term[0] = mul_rn(d, d); term[1] = d; term[2] = mul_rn(di, di); term[3] = di;
        hit[0] = hit[1] = hit[2] = 0;
    } else {
        const GT og = (GT)o;
        const GT d = og > t ? sub_rn(og, t) : sub_rn(t, og);           // :206
        const GT r1 = div_rn(og, t), r2 = div_rn(t, og);               // :217
        const GT mr = r1 > r2 ? r1 : r2;
        const GT io = (GT)__fdiv_rn(1.0f, o);                          // :232 output ** (-1): float32, whatever the target is
        const GT it = div_rn((GT)1.0, t);                              // :233
        const GT di = io > it ? sub_rn(io, it) : sub_rn(it, io);
        term[0] = mul_rn(d, d); term[1] = div_rn(d, t); term[2] = mul_rn(di, di); term[3] = di;
        hit[0] = mr < (GT)1.25; hit[1] = mr < (GT)1.5625; hit[2] = mr < (GT)1.953125;     // :218-220
    }
    return true;
}

// The ground truth as stored (GS) -> its value in the arithmetic type (GT): the identity, or, for the samples of a KITTI
// 16-bit depth PNG, data_read.py:223 `png / 256.` in float64 -- exact, so a ground truth read from its files costs 2 B/px
// and no float64 copy of it exists
template <typename GT, typename GS>
__device__ __forceinline__ GT gt_value(GS s)
{
    if constexpr (std::is_same<GT, GS>::value) return s;
    else {
        static_assert(std::is_same<GT, double>::value && std::is_same<GS, uint16_t>::value, "u16 samples are read as float64");
        return (double)s * (1.0 / 256);
    }
}

// A crop window of the frames (WIN instances, dtfill_eval_sampled: eval_NYU.py:202-207 scores pred[6:234, 8:312]): pixel i
// of the window in its raster order is pixel (r0 + i / cw) * W + c0 + i % cw of a frame of frame_px pixels.  The terms of
// the window's valid pixels are then compacted in the order numpy's boolean index of the cropped view gives them.
struct K4xWindow {
    long frame_px;
    int W, r0, c0, cw;
    __device__ __forceinline__ long at(long i) const
    {
        const int y = (int)i / cw;
        return (long)(r0 + y) * W + c0 + ((int)i - y * cw);
    }
};

// npx: pixels per frame, or per window (WIN); the term arrays hold npx entries per frame either way
template <typename GT, int MODE, typename GS = GT, bool WIN = false>
__global__ void __launch_bounds__(K4X_THREADS) k4x_compact(const float* __restrict__ pred, const GS* __restrict__ gt, long npx,
                                                            GT* __restrict__ terms /*[frames][4][npx]*/,
                                                            int* __restrict__ counts /*[frames][4]*/, const K4xWindow win)
{
    __shared__ int wtot[K4X_THREADS / 32], wbase[K4X_THREADS / 32];
    __shared__ int hits[3];
    const int b = blockIdx.x, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    auto px = [&](long i) -> long { if constexpr (WIN) return win.at(i); else return i; };
    const float* p = pred + (long)b * (WIN ? win.frame_px : npx);
    const GS* g = gt + (long)b * (WIN ? win.frame_px : npx);
    GT* tb = terms + (long)b * 4 * npx;
    const long seg = ((npx + K4X_THREADS - 1) / K4X_THREADS) * 32;     // pixels per warp, a multiple of 32
    const long i0 = min(npx, wid * seg), i1 = min(npx, i0 + seg);
    if (threadIdx.x < 3) hits[threadIdx.x] = 0;
    // pass 1: valid pixels per warp
    int cnt = 0;
    for (long c = i0; c < i1; c += 32) {
        const long i = c + lane;
        const bool v = i < i1 && (p[px(i)] > 0.01f) && (gt_value<GT>(g[px(i)]) > (GT)0.01);     // u16: s >= 3
        cnt += __popc(__ballot_sync(0xffffffffu, v));
    }
    if (lane == 0) wtot[wid] = cnt;
    __syncthreads();
    if (wid == 0) {
        const int c = wtot[lane];
        int inc = c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += o; }
        wbase[lane] = inc - c;
        if (lane == 31) counts[4 * b] = inc;
    }
    __syncthreads();
    // pass 2: terms of the valid pixels at their raster rank
    int run = wbase[wid];
    int h0 = 0, h1 = 0, h2 = 0;
    for (long c = i0; c < i1; c += 32) {
        const long i = c + lane;
        GT term[4] = {0, 0, 0, 0};
        int hit[3] = {0, 0, 0};
        const bool v = i < i1 && metric_terms<GT, MODE>(p[px(i)], gt_value<GT>(g[px(i)]), term, hit);
        const uint32_t m = __ballot_sync(0xffffffffu, v);
        if (v) {
            const long k = run + __popc(m & lanemask_lt());
            tb[k] = term[0]; tb[npx + k] = term[1]; tb[2 * npx + k] = term[2]; tb[3 * npx + k] = term[3];
            h0 += hit[0]; h1 += hit[1]; h2 += hit[2];
        }
        run += __popc(m);
    }
    if (MODE == 1) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            h0 += __shfl_xor_sync(0xffffffffu, h0, d); h1 += __shfl_xor_sync(0xffffffffu, h1, d);
            h2 += __shfl_xor_sync(0xffffffffu, h2, d);
        }
        if (lane == 0) { atomicAdd(&hits[0], h0); atomicAdd(&hits[1], h1); atomicAdd(&hits[2], h2); }
    }
    __syncthreads();
    if (threadIdx.x < 3) counts[4 * b + 1 + threadIdx.x] = hits[threadIdx.x];
}

// numpy's sum of a leaf (n <= 128 elements)
template <typename GT>
__device__ __forceinline__ GT k4x_leaf_sum(const GT* __restrict__ a, int n)
{
    if (n < 8) {
        GT r = (GT)0;
        for (int i = 0; i < n; ++i) r = r + a[i];
        return r;
    }
    GT r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = a[j];
    int i = 8;
    for (; i < n - (n % 8); i += 8) {
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = r[j] + a[i + j];
    }
    GT res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));     // additions only: nothing to contract
    for (; i < n; ++i) res = res + a[i];
    return res;
}

constexpr int K4X_RTHREADS = 256;

template <typename GT>
__global__ void __launch_bounds__(K4X_RTHREADS) k4x_reduce(const GT* __restrict__ terms, const int* __restrict__ counts, long npx,
                                                            int mode, int* __restrict__ leaf_start /*[frames][npx/64 + 2]*/,
                                                            GT* __restrict__ leaf_sum /*[frames][4][npx/64 + 2]*/,
                                                            double* __restrict__ per_frame /*[frames][9]*/)
{
    __shared__ int nleaves;
    __shared__ GT total[4];
    const int b = blockIdx.x;
    const int n = counts[4 * b];
    const long maxl = npx / 64 + 2;
    int* ls = leaf_start + (long)b * maxl;
    GT* lsum = leaf_sum + (long)b * 4 * maxl;
    const GT* tb = terms + (long)b * 4 * npx;
    // the leaves of numpy's recursion, left to right (every leaf but a lone root has 64 < length <= 128)
    if (threadIdx.x == 0) {
        int nl = 0;
        int slo[40], slen[40], sp = 0;
        slo[0] = 0; slen[0] = n;
        while (sp >= 0) {
            const int lo = slo[sp], len = slen[sp];
            --sp;
            if (len <= 128) { ls[nl++] = lo; continue; }
            int n2 = len / 2;
            n2 -= n2 % 8;
            ++sp; slo[sp] = lo + n2; slen[sp] = len - n2;      // right half (handled after the left one)
            ++sp; slo[sp] = lo; slen[sp] = n2;
        }
        ls[nl] = n;
        nleaves = nl;
    }
    __syncthreads();
    const int nl = nleaves;
    for (int l = threadIdx.x; l < nl; l += K4X_RTHREADS) {
        const int lo = ls[l], len = ls[l + 1] - lo;
#pragma unroll
        for (int k = 0; k < 4; ++k) lsum[k * maxl + l] = k4x_leaf_sum<GT>(tb + k * npx + lo, len);
    }
    __syncthreads();
    // the tree: sum(node) = sum(left) + sum(right), leaves consumed left to right; one thread per term array
    if (threadIdx.x < 4) {
        const GT* lv = lsum + threadIdx.x * maxl;
        int li = 0;
        int slen[40], stage[40], sp = 0;
        GT left[40];
        GT ret = (GT)0;
        slen[0] = n; stage[0] = 0;
        while (sp >= 0) {
            const int len = slen[sp];
            if (len <= 128) { ret = lv[li++]; --sp; continue; }
            int n2 = len / 2;
            n2 -= n2 % 8;
            if (stage[sp] == 0) { stage[sp] = 1; ++sp; slen[sp] = n2; stage[sp] = 0; }
            else if (stage[sp] == 1) { left[sp] = ret; stage[sp] = 2; ++sp; slen[sp] = len - n2; stage[sp] = 0; }
            else { ret = left[sp] + ret; --sp; }
        }
        total[threadIdx.x] = ret;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        // np.mean: the sum divided by the count in the arrays' dtype (evaluation.py:94-96, :119-120 / :208-210, :235-236)
        const GT cnt = (GT)n;
        const GT mse = div_rn(total[0], cnt), mae = div_rn(total[1], cnt), imse = div_rn(total[2], cnt), imae = div_rn(total[3], cnt);
        double* o = per_frame + (long)b * 9;
        o[0] = (double)mse;
        o[1] = sqrt((double)mse);                  // math.sqrt of the mean
        o[2] = (double)mae;
        // evaluation.py:119 takes np.sqrt of the mean (the mean's dtype), :235 math.sqrt (float64)
        o[3] = mode == 0 ? (double)sqrt_rn(imse) : sqrt((double)imse);
        o[4] = (double)imae;
        const double dn = (double)n;               // np.mean of a boolean array accumulates in float64: exact counts
        o[5] = mode == 0 ? 0.0 : (double)counts[4 * b + 1] / dn;
        o[6] = mode == 0 ? 0.0 : (double)counts[4 * b + 2] / dn;
        o[7] = mode == 0 ? 0.0 : (double)counts[4 * b + 3] / dn;
        o[8] = dn;
    }
}

// column sums of per_frame over the batch (the running totals of eval.py:212-232), as k4_metrics_final computes them
__global__ void __launch_bounds__(32) k4x_sums(const double* __restrict__ per_frame, int B, double* __restrict__ sums, int accumulate)
{
    if (threadIdx.x < 10) {
        double s = 0.0;
        if (threadIdx.x < 9)
            for (int b = 0; b < B; ++b) s += per_frame[(long)b * 9 + threadIdx.x];
        else
            s = (double)B;
        sums[threadIdx.x] = accumulate ? sums[threadIdx.x] + s : s;
    }
}

}  // namespace dtfill
