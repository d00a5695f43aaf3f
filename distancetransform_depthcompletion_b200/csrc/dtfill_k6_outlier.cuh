// dtfill_k6_outlier.cuh -- K6: KITTI outlier filter (data_read.py:103-128)
#pragma once
#include "dtfill_common.cuh"

namespace dtfill {

// ------------------------------------------------------------------------------------------------------
// K6: KITTI outlier filter, data_read.py:103-128 (SURVEY.md 8 f-2): sum and count over the 7 x 7 diamond
// (cv2.filter2D, default border BORDER_REFLECT_101), average = sum / (count + 1e-5) in float64 (the reference's
// valid_pixels array is float64), a point more than 1.0 m FARTHER than the local average is dropped.  A dropped depth
// becomes a zero of its own sign: x * (1 - 1) in float64 (:128) gives -0.0 for a negative x.
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int reflect101(int i, int n) {
    if (n == 1) return 0;
    while (i < 0 || i >= n) i = i < 0 ? -i : 2 * (n - 1) - i;
    return i;
}

// The filter's verdict for one pixel with value x at (y, x_) of a frame: true = dropped.  BORDER: the window crosses
// the frame edge (reflected indices); kept out of line, it is rare.
template <bool BORDER>
__device__ __forceinline__ bool k6_verdict(const float* __restrict__ frame, int H, int W, int y, int x_, float x)
{
    constexpr int R = 3;
    float sum = 0.f;                       // float32 like cv2.filter2D(sparse_lidar, -1, ...)
    int cnt = 0;                           // the float64 filter of valid_pixels (np.float) counts exactly
#pragma unroll
    for (int dy = -R; dy <= R; ++dy) {
        const int w = R - (dy < 0 ? -dy : dy);
        const float* row = frame + (long)(BORDER ? reflect101(y + dy, H) : y + dy) * W;
#pragma unroll
        for (int dx = -R; dx <= R; ++dx) {
            if (dx < -w || dx > w) continue;
            const float v = __ldg(row + (BORDER ? reflect101(x_ + dx, W) : x_ + dx));
            sum += v;
            cnt += v > 0.1f ? 1 : 0;       // data_read.py:116
        }
    }
    const double aveg = (double)sum / ((double)cnt + 0.00001);         // data_read.py:123
    return ((double)x - aveg) > 1.0;                                   // :125
}
__device__ __noinline__ bool k6_verdict_border(const float* __restrict__ frame, int H, int W, int y, int x_, float x) {
    return k6_verdict<true>(frame, H, W, y, x_, x);
}
__device__ __forceinline__ float k6_dropped(float x) { return __uint_as_float(__float_as_uint(x) & 0x80000000u); }
__device__ __forceinline__ bool k6_is_outlier(const float* __restrict__ frame, int H, int W, int y, int x_, float x) {
    if (y >= 3 && y < H - 3 && x_ >= 3 && x_ < W - 3) return k6_verdict<false>(frame, H, W, y, x_, x);
    return k6_verdict_border(frame, H, W, y, x_, x);
}

// A pixel holding +-0 comes out as it went in whatever its neighbourhood holds (x * (1 - outlier), :128), and a
// LiDAR frame is ~95 % zeros: a thread streams 4 pixels (128-bit load and store) and the 25-tap diamond -- straight
// from global memory through L1 -- is only evaluated for the non-zero ones.  Those are dealt out evenly over the warp
// (VEC: W % 4 == 0, 16-byte aligned): the warp's non-zero pixels form a list ordered by (element, lane) out of four
// ballots, lane l takes entries l, l + 32, ..., fetches the pixel's value and position from its owner by shuffle and
// hands the verdict back through a warp-wide OR.  A beam row (a quarter of its pixels set) then costs a warp two rounds
// of the window code with every lane busy instead of four rounds with a third of them (0.54 -> 0.35 ms per 256 frames).
template <bool VEC>
__global__ void __launch_bounds__(256) k6_outlier_removal(const float* __restrict__ in, int H, int W, long ngroups,
                                                           float* __restrict__ out)
{
    const long g = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (VEC) {
        const int lane = threadIdx.x & 31;
        const bool live = g < ngroups;                                 // whole warps stay for the shuffles
        const int gpr = W >> 2;                                        // groups per row
        const long row = live ? g / gpr : 0;
        const int x0 = live ? (int)(g - row * gpr) * 4 : 0;
        const long frame = row / H;
        const int y = (int)(row - frame * H);
        float4 v = live ? *reinterpret_cast<const float4*>(in + g * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
        const uint32_t m0 = __ballot_sync(0xffffffffu, (__float_as_uint(v.x) << 1) != 0u);
        const uint32_t m1 = __ballot_sync(0xffffffffu, (__float_as_uint(v.y) << 1) != 0u);
        const uint32_t m2 = __ballot_sync(0xffffffffu, (__float_as_uint(v.z) << 1) != 0u);
        const uint32_t m3 = __ballot_sync(0xffffffffu, (__float_as_uint(v.w) << 1) != 0u);
        const int c0 = __popc(m0), c1 = c0 + __popc(m1), c2 = c1 + __popc(m2), total = c2 + __popc(m3);
        uint32_t d0 = 0, d1 = 0, d2 = 0, d3 = 0;                       // owners whose element 0..3 is dropped
        const uint32_t flo = (uint32_t)(frame & 0xffffffffu), fhi = (uint32_t)(frame >> 32);
#pragma unroll 1
        for (int j0 = 0; j0 < total; j0 += 32) {
            const int j = j0 + lane;
            const bool have = j < total;
            const int e = !have ? 0 : (j < c0 ? 0 : (j < c1 ? 1 : (j < c2 ? 2 : 3)));
            const int r = j - (e == 0 ? 0 : (e == 1 ? c0 : (e == 2 ? c1 : c2)));
            const uint32_t me = e == 0 ? m0 : (e == 1 ? m1 : (e == 2 ? m2 : m3));
            const int src = have ? (int)__fns(me, 0, r + 1) : 0;      // lane holding the r-th set bit
            const float vx = __shfl_sync(0xffffffffu, v.x, src), vy = __shfl_sync(0xffffffffu, v.y, src);
            const float vz = __shfl_sync(0xffffffffu, v.z, src), vw = __shfl_sync(0xffffffffu, v.w, src);
            const int sy = __shfl_sync(0xffffffffu, y, src), sx0 = __shfl_sync(0xffffffffu, x0, src);
            const uint32_t slo = __shfl_sync(0xffffffffu, flo, src), shi = __shfl_sync(0xffffffffu, fhi, src);
            bool drop = false;
            if (have) {
                const float x = e == 0 ? vx : (e == 1 ? vy : (e == 2 ? vz : vw));
                const long fsrc = (long)(((unsigned long long)shi << 32) | slo);
                drop = k6_is_outlier(in + fsrc * H * W, H, W, sy, sx0 + e, x);
            }
            const uint32_t bit = drop ? (1u << src) : 0u;
            d0 |= __reduce_or_sync(0xffffffffu, e == 0 ? bit : 0u);
            d1 |= __reduce_or_sync(0xffffffffu, e == 1 ? bit : 0u);
            d2 |= __reduce_or_sync(0xffffffffu, e == 2 ? bit : 0u);
            d3 |= __reduce_or_sync(0xffffffffu, e == 3 ? bit : 0u);
        }
        if (!live) return;
        if ((d0 >> lane) & 1u) v.x = k6_dropped(v.x);
        if ((d1 >> lane) & 1u) v.y = k6_dropped(v.y);
        if ((d2 >> lane) & 1u) v.z = k6_dropped(v.z);
        if ((d3 >> lane) & 1u) v.w = k6_dropped(v.w);
        st_stream_v4(out + g * 4, __float_as_uint(v.x), __float_as_uint(v.y), __float_as_uint(v.z), __float_as_uint(v.w));
    } else {
        if (g >= ngroups) return;
        const long row = g / W;
        const int x0 = (int)(g - row * W);
        const long frame = row / H;
        const int y = (int)(row - frame * H);
        const float x = in[g];
        out[g] = ((__float_as_uint(x) << 1) != 0u && k6_is_outlier(in + frame * H * W, H, W, y, x0, x)) ? k6_dropped(x) : x;
    }
}

}  // namespace dtfill
