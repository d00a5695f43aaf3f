// dtfill_k1_mask.cuh -- K1: predicates, bit rows, validity mask, row-local compaction (tools.py:8, :22; net.py:131-132; data_read.py:215)
#pragma once
#include <type_traits>

#include "dtfill_common.cuh"

namespace dtfill {

// ------------------------------------------------------------------------------------------------------
// K1 (W % 4 == 0): predicates -> bit rows, per-word source prefix, coarse cells, row counts, validity mask,
// and the row-local compaction of the valid depths (into ws.scratch, which K2 only uses later).
// One warp per row; a lane owns 16 consecutive pixels of every 512-pixel chunk (four 128-bit loads).
// The predicates are evaluated without branches: a > b  <=>  sign(b - a) for IEEE floats (a NaN operand gives
// the canonical positive NaN, i.e. "false", like the comparison), and the sign bits of four differences are
// gathered into a nibble with byte permutes and one multiply.
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t sign_nibble(float t0, float t1, float t2, float t3)
{
    // top bytes of the four floats -> one word -> bits 7,15,23,31 -> nibble (multiply gathers them into 28..31)
    const uint32_t p01 = __byte_perm(__float_as_uint(t0), __float_as_uint(t1), 0x0073);   // [t0.b3, t1.b3, 0, 0]
    const uint32_t p23 = __byte_perm(__float_as_uint(t2), __float_as_uint(t3), 0x0073);
    const uint32_t w = __byte_perm(p01, p23, 0x5410) & 0x80808080u;
    return (w * 0x00204081u) >> 28;
}
// the same, and the four sign bits as bytes 0/1 (the validity mask's bytes: one shift instead of nibble -> multiply -> and)
__device__ __forceinline__ uint32_t sign_nibble_bytes(float t0, float t1, float t2, float t3, uint32_t& bytes01)
{
    const uint32_t p01 = __byte_perm(__float_as_uint(t0), __float_as_uint(t1), 0x0073);
    const uint32_t p23 = __byte_perm(__float_as_uint(t2), __float_as_uint(t3), 0x0073);
    const uint32_t w = __byte_perm(p01, p23, 0x5410) & 0x80808080u;
    bytes01 = w >> 7;
    return (w * 0x00204081u) >> 28;
}

// Sampled input (T = SampledGt, dtfill_eval_sampled): `in` is the whole ground truth, not offset to the sub-batch, and frame
// frame0 + f of the call reads ground-truth frame (frame0 + f) mod fp.gt_frames, so that the frames of several draws share
// one ground truth.  The sample bitmap of k10_sample_bits lies in ws.srcbits, in the layout
// K1 writes its source bits in.  A word is read by the two lanes (or, in the scalar kernel, the warp) that later overwrite
// it, and every read value is consumed before the warp's shuffles / ballots that precede the write.  A pixel keeps its
// ground-truth value when its bit is set and becomes g * 0 otherwise, as `gt * Mask` does (data_read.py:364): -0 for a
// negative g, NaN for a NaN or infinite g (a source, tools.py:8).
__device__ __forceinline__ float sampled_px(float g, uint32_t bit) { return bit ? g : __fmul_rn(g, 0.0f); }
// the 16 bits of the lane's pixels [col, col + 16) of row `row` (col a multiple of 16)
__device__ __forceinline__ uint32_t sample_half(const Workspace& ws, long row, int WW, int col, int W)
{
    return col < W ? (ws.srcbits[row * WW + (col >> 5)] >> (col & 16)) & 0xFFFFu : 0u;
}

// W16: W % 16 == 0 (KITTI 1216, NYU 640): a lane's 16 pixels are inside the row or outside it as a whole.
template <typename T, bool W16>
__global__ void __launch_bounds__(256) k1_mask_rows_v16(const T* __restrict__ in, FrameParams fp, Workspace ws,
                                                         uint8_t* __restrict__ out_mask, float* __restrict__ out_lidar)
{
    DTFILL_TRACE_SCOPE(fp, 0);
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    const int W = fp.W, WW = fp.WW;
    const long nrows = (long)fp.B * fp.H;
    const bool rows32 = nrows < (1l << 31);
    const int nchunks = (W + 511) >> 9;
    const float scut = fp.src_cut, vthr = fp.val_thr;
    float* rowvals = reinterpret_cast<float*>(ws.scratch);
    for (long row = warp; row < nrows; row += nwarps) {
        const T* rp = in + row * W;
        if constexpr (std::is_same<T, SampledGt>::value) {   // row -> (frame, y), y of ground-truth frame f mod gt_frames
            const long frame = rows32 ? (long)((uint32_t)row / (uint32_t)fp.H) : row / fp.H;
            const long g = (long)((uint32_t)(fp.frame0 + frame) % (uint32_t)fp.gt_frames);
            rp = in + (g * fp.H + (row - frame * fp.H)) * W;
        } else if (fp.in_H != fp.H) {                // cropped input frames (uint16 entry): row -> (frame, y)
            const long frame = rows32 ? (long)((uint32_t)row / (uint32_t)fp.H) : row / fp.H;
            rp = in + (frame * fp.in_H + fp.in_crop + (row - frame * fp.H)) * W;
        }
        uint32_t cs = 0, cv = 0;
        // software pipeline over the 512-pixel chunks: the 128-bit loads of the next chunk are issued (volatile
        // asm, so they stay ahead) before the current chunk is processed
        In16<T> nq;
        if (W16) nq.load_all(rp + lane * 16, lane * 16 < W);
        else nq.load(rp + lane * 16, lane * 16, W);
        uint32_t nbits = 0;
        if constexpr (std::is_same<T, SampledGt>::value) nbits = sample_half(ws, row, WW, lane * 16, W);
        for (int ch = 0; ch < nchunks; ++ch) {
            const int col = (ch << 9) + lane * 16;
            float4 q[4];
#pragma unroll
            for (int g = 0; g < 4; ++g) q[g] = nq.get(g);
            const uint32_t bits = nbits;
            if (ch + 1 < nchunks) {
                if (W16) nq.load_all(rp + col + 512, col + 512 < W);
                else nq.load(rp + col + 512, col + 512, W);
                if constexpr (std::is_same<T, SampledGt>::value) nbits = sample_half(ws, row, WW, col + 512, W);
            }
            if constexpr (std::is_same<T, SampledGt>::value) {
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    const uint32_t b4 = bits >> (4 * g);
                    q[g] = make_float4(sampled_px(q[g].x, b4 & 1u), sampled_px(q[g].y, b4 & 2u), sampled_px(q[g].z, b4 & 4u),
                                       sampled_px(q[g].w, b4 & 8u));
                }
            }
            if (out_lidar && col < W) {                  // decoded (uint16) or sampled frame: what the CNN reads as lidar
#pragma unroll
                for (int g = 0; g < 4; ++g)
                    if (W16 || col + 4 * g < W)
                        st_stream_v4(out_lidar + row * W + col + 4 * g, __float_as_uint(q[g].x), __float_as_uint(q[g].y),
                                     __float_as_uint(q[g].z), __float_as_uint(q[g].w));
            }
            uint32_t sb = 0, vb = 0;
            uint32_t m[4];                                   // validity mask bytes of the lane's 16 pixels
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                // tools.py:8: source <=> !(float32(1 - x) > src_thr) <=> !(x < src_cut), src_cut being the smallest
                // float that satisfies the predicate (found on the host, the predicate is monotone in x);
                // tools.py:22: valid <=> x > val_thr
                const uint32_t ns = sign_nibble(__fsub_rn(q[g].x, scut), __fsub_rn(q[g].y, scut), __fsub_rn(q[g].z, scut),
                                                __fsub_rn(q[g].w, scut));                   // bit = x < src_cut
                const uint32_t nv = sign_nibble_bytes(__fsub_rn(vthr, q[g].x), __fsub_rn(vthr, q[g].y),
                                                      __fsub_rn(vthr, q[g].z), __fsub_rn(vthr, q[g].w), m[g]);
                sb |= ns << (4 * g);
                vb |= nv << (4 * g);
            }
            const uint32_t inb = W16 ? (col < W ? 0xFFFFu : 0u)              // pixels of this lane inside the row
                                     : (1u << min(max(W - col, 0), 16)) - 1u;
            sb = ~sb & inb;
            vb &= inb;
            if (out_mask && col < W) {
                if (!W16) {                                  // pixels beyond the row's end are not valid
#pragma unroll
                    for (int g = 0; g < 4; ++g) m[g] = (((vb >> (4 * g)) & 0xFu) * 0x00204081u) & 0x01010101u;
                }
                uint8_t* mp = out_mask + row * W + col;
                if (W16) {
                    st_stream_v4(mp, m[0], m[1], m[2], m[3]);
                } else {
#pragma unroll
                    for (int g = 0; g < 4; ++g)
                        if (col + 4 * g < W) st_stream_u32(mp + 4 * g, m[g]);
                }
            }
            // 32-bit words from the halves of 2 neighbouring lanes
            uint32_t sw = sb << ((lane & 1) * 16);
            sw |= __shfl_xor_sync(0xffffffffu, sw, 1);
            // coarse cells: bit j of the word's nibble = some source among its pixels 8j..8j+7
            const uint32_t cell = ((sw & 0xFFu) != 0) | (((sw & 0xFF00u) != 0) << 1) | (((sw & 0xFF0000u) != 0) << 2) |
                                  (((sw & 0xFF000000u) != 0) << 3);
            // one scan for both counts: sources in the low half, valid pixels in the high half (<= 512 each)
            const uint32_t anybits = __ballot_sync(0xffffffffu, (sb | vb) != 0);
            uint32_t pre = 0, tot = 0;
            if (anybits) {
                const uint32_t c = __popc(sb) | (__popc(vb) << 16);
                uint32_t inc = c;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
                    if (lane >= d) inc += o;
                }
                pre = inc - c;
                tot = __shfl_sync(0xffffffffu, inc, 31);
            }
            const int w = (ch << 4) + (lane >> 1);
            if ((lane & 1) == 0 && w < WW) {
                const long wi = row * WW + w;
                ws.srcbits[wi] = sw;
                ws.wprefix[wi] = (uint16_t)(cs + (pre & 0xFFFFu));
                ws.rowcell[wi] = (uint8_t)cell;
            }
            cs += tot & 0xFFFFu;
            if (tot >> 16) {
                // the lane's valid values, still in registers, go out with predicated stores (a loop over the set
                // bits would run as often as the busiest lane has valid pixels, 7 times on a beam row)
                // (addresses as 32 x 32 + 64 multiply-adds with a run-time multiplier: FMA pipe, not the ALU pipe this
                // kernel saturates)
                const char* dst = reinterpret_cast<const char*>(rowvals + row * W + cv + (pre >> 16));
                uint32_t off = 0;
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    const float vv[4] = {q[g].x, q[g].y, q[g].z, q[g].w};
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const bool p = (vb & (1u << (4 * g + e))) != 0;
                        float* a = reinterpret_cast<float*>(const_cast<char*>(dst) + (uint64_t)off * fp.four);
                        if (p) *a = vv[e];
                        off = p ? off * fp.one + 1u : off;
                    }
                }
                cv += tot >> 16;
            }
        }
        if (lane == 0) {
            ws.rowsrc[row] = cs;
            ws.rowval[row] = cv;
        }
    }
}

// ------------------------------------------------------------------------------------------------------
// K1 for widths that are not a multiple of 4 (no 128-bit row alignment): same outputs, scalar loads + ballots.
// ------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) k1_mask_rows(const T* __restrict__ in, FrameParams fp, Workspace ws,
                                                     uint8_t* __restrict__ out_mask, float* __restrict__ out_lidar)
{
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    const int W = fp.W, WW = fp.WW;
    const long nrows = (long)fp.B * fp.H;
    const bool rows32 = nrows < (1l << 31);
    const bool vec_mask = (W & 3) == 0;
    const uint32_t ltmask = lanemask_lt();
    float* rowvals = reinterpret_cast<float*>(ws.scratch);
    for (long row = warp; row < nrows; row += nwarps) {
        const T* rp = in + row * W;
        if constexpr (std::is_same<T, SampledGt>::value) {   // row -> (frame, y), y of ground-truth frame f mod gt_frames
            const long frame = rows32 ? (long)((uint32_t)row / (uint32_t)fp.H) : row / fp.H;
            const long g = (long)((uint32_t)(fp.frame0 + frame) % (uint32_t)fp.gt_frames);
            rp = in + (g * fp.H + (row - frame * fp.H)) * W;
        } else if (fp.in_H != fp.H) {                // cropped input frames (uint16 entry): row -> (frame, y)
            const long frame = rows32 ? (long)((uint32_t)row / (uint32_t)fp.H) : row / fp.H;
            rp = in + (frame * fp.in_H + fp.in_crop + (row - frame * fp.H)) * W;
        }
        uint32_t cs = 0, cv = 0;
        for (int c0 = 0; c0 < WW; c0 += 16) {
            float x[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                const int col = (c0 + k) * 32 + lane;
                x[k] = col < W ? load_px_stream(rp + col) : 0.0f;
                if constexpr (std::is_same<T, SampledGt>::value)
                    if (col < W) x[k] = sampled_px(x[k], (ws.srcbits[row * WW + c0 + k] >> lane) & 1u);
                if (out_lidar && col < W) out_lidar[row * W + col] = x[k];
            }
            uint32_t mys = 0, mypre = 0;
            uint32_t vq[4];
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                const int col = (c0 + k) * 32 + lane;
                const bool inb = col < W;
                const float d = __fsub_rn(1.0f, x[k]);                 // tools.py:8  1.0 - x  (float32)
                const bool sp = inb && !(d > fp.src_thr);             // value_mask == 0  <=> source
                const bool vp = inb && (x[k] > fp.val_thr);           // tools.py:22 with_value
                const uint32_t sw = __ballot_sync(0xffffffffu, sp);
                const uint32_t vw = __ballot_sync(0xffffffffu, vp);
                if (lane == k) { mys = sw; mypre = cs; }
                if (vp) rowvals[row * W + cv + __popc(vw & ltmask)] = x[k];
                cs += __popc(sw);
                cv += __popc(vw);
                vq[k & 3] = vw;
                if (out_mask) {
                    if (vec_mask) {
                        if ((k & 3) == 3) {
                            const int col4 = (c0 + k - 3) * 32 + lane * 4;
                            if (col4 < W) {
                                const int q = lane >> 3;
                                const uint32_t word = q == 0 ? vq[0] : q == 1 ? vq[1] : q == 2 ? vq[2] : vq[3];
                                const uint32_t nib = (word >> ((lane & 7) * 4)) & 0xFu;
                                st_stream_u32(out_mask + row * W + col4, (nib * 0x00204081u) & 0x01010101u);
                            }
                        }
                    } else if (inb) {
                        out_mask[row * W + col] = (uint8_t)vp;
                    }
                }
            }
            if (lane < 16 && c0 + lane < WW) {
                const long wi = row * WW + c0 + lane;
                ws.srcbits[wi] = mys;
                ws.wprefix[wi] = (uint16_t)mypre;
                ws.rowcell[wi] = (uint8_t)(((mys & 0xFFu) != 0) | (((mys & 0xFF00u) != 0) << 1) |
                                           (((mys & 0xFF0000u) != 0) << 2) | (((mys & 0xFF000000u) != 0) << 3));
            }
        }
        if (lane == 0) {
            ws.rowsrc[row] = cs;
            ws.rowval[row] = cv;
        }
    }
}

}  // namespace dtfill
