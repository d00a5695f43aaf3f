// dtfill_k10_sample.cuh -- K10: the NYU sample mask (data_read.py:360-364) as a bitmap, the step before K1 of dtfill_eval_sampled
#pragma once
#include "dtfill_common.cuh"

namespace dtfill {

// ------------------------------------------------------------------------------------------------------
// `Mask[rows, cols] = 1` for every frame of a batch: one block per frame scatters the frame's (row, col) pairs
// rows[offsets[b] : offsets[b+1]] into a bitmap of 1 bit per pixel, bit (col & 31) of word (b*H + row) * WW + col/32 --
// the layout of K1's source bits, where K1's sampled input kind reads it (dtfill_k1_mask.cuh).  atomicOr, so duplicates
// collapse as they do in the reference's assignment.  The bitmap is cleared on the same stream before the launch.  A frame
// with decreasing offsets or a coordinate outside [0,H) x [0,W) sets nothing out of place and lowers *bad to its index.
// ------------------------------------------------------------------------------------------------------
constexpr int K10_THREADS = 256;

__global__ void __launch_bounds__(K10_THREADS) k10_sample_bits(const int32_t* __restrict__ rows, const int32_t* __restrict__ cols,
                                                               const int64_t* __restrict__ offsets, int H, int W, int WW,
                                                               uint32_t* __restrict__ bits, int* __restrict__ bad)
{
    const int b = blockIdx.x;
    const int64_t lo = offsets[b], hi = offsets[b + 1];
    if (lo < 0 || hi < lo) {
        if (threadIdx.x == 0) atomicMin(bad, b);
        return;
    }
    uint32_t* fb = bits + (size_t)b * H * WW;
    for (int64_t i = lo + threadIdx.x; i < hi; i += K10_THREADS) {
        const int r = rows[i], c = cols[i];
        if ((unsigned)r >= (unsigned)H || (unsigned)c >= (unsigned)W) {
            atomicMin(bad, b);
            continue;
        }
        atomicOr(fb + (size_t)r * WW + (c >> 5), 1u << (c & 31));
    }
}

}  // namespace dtfill
