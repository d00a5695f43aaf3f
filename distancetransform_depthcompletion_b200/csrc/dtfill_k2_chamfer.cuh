// dtfill_k2_chamfer.cuh -- K2: OpenCV's 5x5 chamfer scan with labels on packed 32-bit keys + gather (tools.py:9, :25-27)
#pragma once
#include "dtfill_common.cuh"

namespace dtfill {

// ------------------------------------------------------------------------------------------------------
// K2: the chamfer scan, fast path.  One warp per task; lane l owns columns [l*PPL, (l+1)*PPL) of every row.
// ------------------------------------------------------------------------------------------------------
template <int PPL>
struct Row {
    uint32_t v[PPL];
    uint32_t l1, l2;   // columns -1, -2 (previous lane's last two)
    uint32_t r0, r1;   // columns PPL, PPL+1 (next lane's first two)
};

template <int PPL>
__device__ __forceinline__ uint32_t at(const Row<PPL>& r, int idx) {
    // idx is a compile-time constant after unrolling
    return idx == -2 ? r.l2 : idx == -1 ? r.l1 : idx == PPL ? r.r0 : idx == PPL + 1 ? r.r1 : r.v[idx < 0 ? 0 : (idx >= PPL ? PPL - 1 : idx)];
}

template <int PPL>
__device__ __forceinline__ void fill_row(Row<PPL>& r, uint32_t k) {
#pragma unroll
    for (int i = 0; i < PPL; ++i) r.v[i] = k;
    r.l1 = r.l2 = r.r0 = r.r1 = k;
}

template <int PPL>
__device__ __forceinline__ void refresh_halo(Row<PPL>& r, int lane, uint32_t init_key) {
    const uint32_t a = __shfl_up_sync(0xffffffffu, r.v[PPL - 1], 1);
    const uint32_t b = __shfl_up_sync(0xffffffffu, r.v[PPL - 2], 1);
    const uint32_t c = __shfl_down_sync(0xffffffffu, r.v[0], 1);
    const uint32_t d = __shfl_down_sync(0xffffffffu, r.v[1], 1);
    r.l1 = lane == 0 ? init_key : a;
    r.l2 = lane == 0 ? init_key : b;
    r.r0 = lane == 31 ? init_key : c;
    r.r1 = lane == 31 ? init_key : d;
}

// Carry entering this lane from the lanes before it (DIR=+1, forward scan) or after it (DIR=-1, backward
// scan).  e = this lane's outgoing value (cleared key).  Works in a widened dist:14|label:18 form so that
// adding up to 31*PPL columns cannot overflow.  Ties keep the nearer lane (OpenCV: the left neighbour is
// the last candidate compared, so a value already held wins).
template <int PPL, int DIR>
__device__ __forceinline__ uint32_t lane_carry(uint32_t e, int lane, uint32_t clamp_dist)
{
    uint32_t E = ((e >> DSH) << OSH) | (e & LMASK);
    {   // distance 1: the neighbouring lane
        const uint32_t o = DIR > 0 ? __shfl_up_sync(0xffffffffu, E, 1) : __shfl_down_sync(0xffffffffu, E, 1);
        const uint32_t t = o + (uint32_t(PPL) << OSH);
        E = ((t | LMASK) < E) ? t : E;
    }
    // a value carried over d >= 2 lanes is at least 2*PPL; it can only win where a lane's own value is larger than
    // that, which never happens in densely sampled tiles: one warp-wide maximum decides whether to go on
    if (__reduce_max_sync(0xffffffffu, E >> OSH) >= 2u * PPL) {
#pragma unroll
        for (int d = 2; d < 32; d <<= 1) {
            const uint32_t o = DIR > 0 ? __shfl_up_sync(0xffffffffu, E, d) : __shfl_down_sync(0xffffffffu, E, d);
            const uint32_t t = o + (uint32_t(d * PPL) << OSH);
            E = ((t | LMASK) < E) ? t : E;
        }
    }
    const uint32_t cin = DIR > 0 ? __shfl_up_sync(0xffffffffu, E, 1) : __shfl_down_sync(0xffffffffu, E, 1);
    const uint32_t cd = min(cin >> OSH, clamp_dist);
    uint32_t key = (cd << DSH) | (1u << OSH) | (cin & LMASK);
    const bool edge = DIR > 0 ? (lane == 0) : (lane == 31);
    if (edge) key = (clamp_dist << DSH) | (1u << OSH);
    return key;
}

__device__ __forceinline__ void cp_async8(uint32_t smem_addr, const void* gptr) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_addr), "l"(gptr) : "memory");
}
// forward-state scratch is written once and read once, a whole pass later: keep it out of L1 (L2 only)
__device__ __forceinline__ void st_scratch_v4(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.global.cg.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void st_scratch_v2(void* p, uint32_t a, uint32_t b) {
    asm volatile("st.global.cg.v2.u32 [%0], {%1, %2};" ::"l"(p), "r"(a), "r"(b) : "memory");
}
// One row of the forward state (128 * PPL contiguous bytes of scratch) -> shared memory as a single bulk-copy (TMA)
// transaction; completion is signalled on an mbarrier that the whole warp waits on, phase by phase.
__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void bulk_row_to_smem(uint32_t smem_dst, const void* gsrc, uint32_t bytes, uint32_t mbar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_dst), "l"(gsrc), "r"(bytes), "r"(mbar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity) {
    uint32_t done = 0;
    while (!done)
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(mbar), "r"(parity) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// dist field of a key as float, on the FMA pipe (the ALU pipe is the one this kernel saturates):
// (key >> 21) + 2^23 as the high half of a multiply-add, then the float with that bit pattern minus 2^23.
__device__ __forceinline__ float key_dist_f32(uint32_t key, uint32_t mul_dist) {
    uint32_t t;
    asm("mad.hi.u32 %0, %1, %2, %3;" : "=r"(t) : "r"(key), "r"(mul_dist), "r"(0x4B000000u));
    return __uint_as_float(t) - 8388608.0f;
}

// Raw words holding this lane's PPL source bits of one row, fetched one row ahead of their use.
struct RowBits {
    uint32_t a, b, c, pre, base;
};

template <int PPL>
__device__ __forceinline__ RowBits fetch_row_bits(const uint32_t* __restrict__ bits_f, const uint16_t* __restrict__ pre_f,
                                                  const uint32_t* __restrict__ rowbase, int WW, int x0, int y)
{
    RowBits r;
    const int w = x0 >> 5;
    const uint32_t* br = bits_f + (long)y * WW;
    r.a = w < WW ? br[w] : 0u;
    r.b = w + 1 < WW ? br[w + 1] : 0u;
    r.c = (PPL > 33 && w + 2 < WW) ? br[w + 2] : 0u;
    r.pre = w < WW ? (uint32_t)pre_f[(long)y * WW + w] : 0u;
    r.base = rowbase[y];
    return r;
}

// bit i of `bits` = column x0+i is a source; rank = 1-based raster rank of the first source of this lane
template <int PPL>
struct LaneBits { typedef uint64_t type; };
template <> struct LaneBits<10> { typedef uint32_t type; };
template <> struct LaneBits<20> { typedef uint32_t type; };

template <int PPL>
__device__ __forceinline__ void decode_row_bits(const RowBits& r, int x0, typename LaneBits<PPL>::type& bits,
                                                uint32_t& rank)
{
    const int sh = x0 & 31;
    if (sizeof(typename LaneBits<PPL>::type) == 4) {
        bits = __funnelshift_r(r.a, r.b, sh) & ((1u << (PPL & 31)) - 1u);     // PPL <= 32 bits from two words
    } else {
        uint64_t lo = ((uint64_t)r.b << 32) | r.a;
        lo >>= sh;
        if (PPL > 33 && sh) lo |= (uint64_t)r.c << (64 - sh);
        bits = (typename LaneBits<PPL>::type)(lo & ((PPL >= 64) ? ~0ull : ((1ull << PPL) - 1ull)));
    }
    rank = r.base + r.pre + __popc(r.a & ((1u << sh) - 1u)) + 1u;
}


// ------------------------------------------------------------------------------------------------------
// The 7 (forward) / 1 + 7 (backward) candidates of a pixel.  All candidates are full keys with distinct order
// fields, so their minimum is OpenCV's "first strictly smaller candidate wins" however it is grouped.  The ALU pipe
// (VIADDMNMX, VIMNMX3, LOP3: one warp instruction per 2 cycles and SM sub-partition) is what the scan saturates;
// the FMA pipe (IMAD) runs beside it at the same rate (profiles/ubench/pipes.cu: 3.8 warp instructions per clock
// and SM for a 1:1 mix against 1.9 for either alone).  Three of the forward additions (two backward) are plain IMADs
// whose results meet in a 3-input minimum; DESIGN.md §5 records the other splits that were measured.
// ------------------------------------------------------------------------------------------------------
// Resident warps per SM the PPL = 20 instance is compiled for: its register budget (more warps spill).
constexpr int K2_WARPS_PPL20 = 20;

template <int PPL>
__device__ __forceinline__ uint32_t stencil_fwd(const Row<PPL>& A /*row y-1*/, const Row<PPL>& Bq /*row y-2*/, int i, uint32_t one)
{
    const uint32_t b0 = at(Bq, i - 1), b1 = at(Bq, i + 1);
    const uint32_t a0 = at(A, i - 2), a1 = at(A, i - 1), a2 = at(A, i), a3 = at(A, i + 1), a4 = at(A, i + 2);
    // OpenCV's order: (-2,-1) (-2,+1) (-1,-2) (-1,-1) (-1,0) (-1,+1) (-1,+2); orders 0,2,..,12 (even: see header)
    const uint32_t m0 = __viaddmin_u32(b1, KC(3, 2), b0 * one + KC(3, 0));
    const uint32_t m1 = __viaddmin_u32(a1, KC(2, 6), a0 * one + KC(3, 4));
    uint32_t m2 = __viaddmin_u32(a3, KC(2, 10), a2 * one + KC(1, 8));
    m2 = __viaddmin_u32(a4, KC(3, 12), m2);
    return __vimin3_u32(m0, m1, m2);
}

template <int PPL>
__device__ __forceinline__ uint32_t stencil_bwd(uint32_t own /*forward key, order <= 1*/, const Row<PPL>& A /*row y+1*/,
                                                const Row<PPL>& Bq /*row y+2*/, int i, uint32_t one)
{
    const uint32_t b0 = at(Bq, i + 1), b1 = at(Bq, i - 1);
    const uint32_t a0 = at(A, i + 2), a1 = at(A, i + 1), a2 = at(A, i), a3 = at(A, i - 1), a4 = at(A, i - 2);
    // own value first, then (+2,+1) (+2,-1) (+1,+2) (+1,+1) (+1,0) (+1,-1) (+1,-2); orders 2,4,..,14
    uint32_t m0 = __viaddmin_u32(b0, KC(3, 2), own);
    m0 = __viaddmin_u32(b1, KC(3, 4), m0);
    const uint32_t m1 = __viaddmin_u32(a1, KC(2, 8), a0 * one + KC(3, 6));
    uint32_t m2 = __viaddmin_u32(a3, KC(2, 12), a2 * one + KC(1, 10));
    m2 = __viaddmin_u32(a4, KC(3, 14), m2);
    return __vimin3_u32(m0, m1, m2);
}

template <int PPL, bool PAD, bool WANT_LBL, bool VEC>
__global__ void __launch_bounds__(32, (PPL >= 38 ? 12 : (PPL >= 20 ? K2_WARPS_PPL20 : 32))) k2_chamfer(FrameParams fp, Workspace ws, float* __restrict__ out_depth,
                                                  float* __restrict__ out_dt, int32_t* __restrict__ out_lbl, int my_kind)
{
    // Transposition buffer for the keys of an output row.  Keeping shared memory small matters: what is left of the
    // 228 KB is the L1 that serves the depth_list gather.
    __shared__ __align__(16) uint32_t stage_smem[32 * PPL];
    uint32_t* stage = stage_smem;
    __shared__ __align__(16) uint2 fwdbuf[16 * PPL];      // forward keys of the next row to scan, [j][lane]
    __shared__ __align__(8) uint64_t fwdbar;              // completion of the bulk copy into fwdbuf

    const Task task = ws.tasks[blockIdx.x];      // slot-major: blockIdx = slot * B + frame, longest tasks first
    if (task.kind != my_kind && !(task.kind == TASK_NOSRC && my_kind == TASK_CHAMFER)) return;
    DTFILL_TRACE_SCOPE(fp, 2);
    const int lane = threadIdx.x;
    const int H = fp.H, W = fp.W, WW = fp.WW;
    const int b = task.frame;
    const long fpx = (long)b * H * W;

    if (task.kind == TASK_NOSRC) {
        // no source anywhere: OpenCV leaves dt at 65533 and lbl at 0; depth_list[0-1] is numpy's last element
        const int nval = ws.counts[2 * b + 1];
        const float last = ws.dlist[fpx + (nval > 0 ? nval - 1 : 0)];
        for (long i = (long)task.r0 * W + lane; i < (long)task.r1 * W; i += 32) {
            out_depth[fpx + i] = last;
            if (out_dt) out_dt[fpx + i] = UNREACHED_DT;
            if (WANT_LBL) out_lbl[fpx + i] = 0;
        }
        return;
    }

    const int x0 = task.clo + lane * PPL;        // first image column of this lane
    const int xl = lane * PPL;                   // same, relative to the tile
    const uint32_t init_key = (uint32_t)fp.init_dist << DSH;
    const uint32_t clamp_dist = 2047u - PPL - 1u;
    const uint32_t* bits_f = ws.srcbits + (long)b * H * WW;
    const uint16_t* pre_f = ws.wprefix + (long)b * H * WW;
    const uint32_t* rowbase = ws.rowsrc + (long)b * H;
    constexpr int VW = (PPL % 4 == 0) ? 4 : 2;   // keys per scratch vector
    uint2* scr = reinterpret_cast<uint2*>(ws.scratch) + (long)task.scratch_off * 16;   // 32*PPL keys per row

    Row<PPL> ra, rb;
    fill_row(ra, init_key);
    fill_row(rb, init_key);

    // ---------------- forward pass: rows lo .. hi-1 ----------------
    RowBits nextbits = fetch_row_bits<PPL>(bits_f, pre_f, rowbase, WW, x0, task.fstart);
    auto fwd_step = [&](const Row<PPL>& A /*row y-1*/, Row<PPL>& Bq /*row y-2 in, row y out*/, int y) {
        typename LaneBits<PPL>::type bits; uint32_t rank;
        decode_row_bits<PPL>(nextbits, x0, bits, rank);
        nextbits = fetch_row_bits<PPL>(bits_f, pre_f, rowbase, WW, x0, min(y + 1, task.hi - 1));   // one row ahead
        if (lane < 2 && y + 4 < task.hi) {           // bit row and prefixes four rows ahead -> L2
            asm volatile("prefetch.global.L2 [%0];" ::"l"(bits_f + (long)(y + 4) * WW + (x0 >> 5) + lane * 32));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(pre_f + (long)(y + 4) * WW + (x0 >> 5) + lane * 32));
        }
        uint32_t c[PPL];
#pragma unroll
        for (int i = 0; i < PPL; ++i) c[i] = stencil_fwd<PPL>(A, Bq, i, fp.one);
        if (__any_sync(0xffffffffu, bits != 0)) {                         // sources: dist 0, own raster rank
#pragma unroll
            for (int i = 0; i < PPL; ++i) {
                const bool s = (bits & ((typename LaneBits<PPL>::type)1 << i)) != 0;
                c[i] = s ? rank : c[i];
                rank += s ? 1u : 0u;
            }
        }
        // in-lane scan: T[x] = min(c[x], T[x-1] + 1); the left neighbour is OpenCV's last candidate (order 14).
        // Two independent half-lane chains (twice the instruction-level parallelism of one chain of PPL dependent
        // steps), joined afterwards: a value entering the second half from the first is one more "left" candidate
        // (order 1, loses ties against anything the second half holds itself)
        constexpr int HF = PPL / 2;
        uint32_t u = c[0] & ORDCLR, u2 = c[HF] & ORDCLR;
        c[0] = u; c[HF] = u2;
#pragma unroll
        for (int i = 1; i < PPL - HF; ++i) {
            if (i < HF) { u = __viaddmin_u32(u, KC(1, 14), c[i]) & ORDCLR; c[i] = u; }
            u2 = __viaddmin_u32(u2, KC(1, 14), c[HF + i]) & ORDCLR; c[HF + i] = u2;
        }
        const uint32_t e = __viaddmin_u32(u | (1u << OSH), uint32_t(PPL - HF) << DSH, u2) & ORDCLR;    // lane's last column
        const uint32_t cin = lane_carry<PPL, +1>(e, lane, clamp_dist);
        const uint32_t cin2 = __viaddmin_u32(cin, uint32_t(HF) << DSH, u) | (1u << OSH);               // column HF-1, final
#pragma unroll
        for (int i = 0; i < PPL; ++i) {
            uint32_t t = i < HF ? __viaddmin_u32(cin, uint32_t(i + 1) << DSH, c[i])
                                : __viaddmin_u32(cin2, uint32_t(i - HF + 1) << DSH, c[i]);   // order bit 0/1 stays (see header)
            if (PAD && x0 + i >= W) t = init_key;
            Bq.v[i] = t;
        }
        refresh_halo(Bq, lane, init_key);
        // forward state -> scratch, [vector j][lane] so that every store instruction is fully coalesced; the rows of
        // the upper halo are never read back (the backward pass ends at r0)
        if (y >= task.r0) {
            char* dst = reinterpret_cast<char*>(scr) + (long)(y - task.lo) * (128 * PPL) + lane * (4 * VW);
#pragma unroll
            for (int j = 0; j < PPL / VW; ++j) {
                if (VW == 4) st_scratch_v4(dst + j * 512, Bq.v[4 * j], Bq.v[4 * j + 1], Bq.v[4 * j + 2], Bq.v[4 * j + 3]);
                else st_scratch_v2(dst + j * 256, Bq.v[2 * j], Bq.v[2 * j + 1]);
            }
        }
    };

    // one copy of the step in the instruction stream (the unrolled step is ~13 KB of code); the two live rows
    // are rotated with register moves, which go to the otherwise idle FMA pipe
#pragma unroll 1
    for (int y = task.fstart; y < task.hi; ++y) {
        fwd_step(ra, rb, y);
        const Row<PPL> t = ra; ra = rb; rb = t;
    }

    // ---------------- backward pass: rows hi-1 .. r0 ----------------
    // The forward keys of row y-1 are copied scratch -> fwdbuf while row y is being scanned: no registers, no exposed
    // latency.  With 4-key vectors (PPL % 4 == 0) the row is one bulk copy (TMA) issued by lane 0 and signalled on an
    // mbarrier; otherwise every lane copies its own keys with 8-byte cp.async.  (The depth gather is NOT done with
    // cp.async: 4-byte LDGSTS cost 8 LSU cycles each and 20-38 of them per row step saturate the LSU -- measured.)
    fill_row(ra, init_key);
    fill_row(rb, init_key);
    const float* dl = ws.dlist + fpx;
    // depth_list is the one buffer of the path that is read at random and more than once (21 MB per batch of 256 KITTI
    // frames); K1b writes it and the gather below reads it with plain stores and loads
    const char* dlm1_bytes = reinterpret_cast<const char*>(dl - 1);       // depth_list[lbl - 1]
    // output addressing that does not depend on the row: which 4-pixel groups of the transposed row this lane
    // writes (inside [c0,c1)), and where
    constexpr int NJ = (32 * PPL + 127) / 128;
    uint32_t okmask = 0;
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
        const int lc = (j * 32 + lane) * 4, col = task.clo + lc;
        if (lc < 32 * PPL && col >= task.c0 && col < task.c1) okmask |= 1u << j;
    }
    const long colbase = fpx + task.clo + lane * 4;
    const uint4* sread = reinterpret_cast<const uint4*>(&stage[lane * 4]);
    uint2* swrite = reinterpret_cast<uint2*>(&stage[xl]);
    const uint32_t fwdbuf_lane = (uint32_t)__cvta_generic_to_shared(fwdbuf) + lane * (4 * VW);

    constexpr bool TMA_ROWS = VW == 4;
    const uint32_t fwdbar_a = (uint32_t)__cvta_generic_to_shared(&fwdbar);
    const uint32_t fwdbuf_a = (uint32_t)__cvta_generic_to_shared(fwdbuf);
    if (TMA_ROWS) {
        if (lane == 0) mbar_init(fwdbar_a, 1);
        // The forward rows were written with ordinary stores (generic proxy); the bulk copies below read them through
        // the async proxy.  Without this fence the copy of the rows written last (hi - 1, hi - 2: the first ones the
        // backward pass needs) can overtake their stores -- seen as wrong values in the bottom rows of a few frames per
        // thousand when four batches were in flight.  Every lane fences its own stores, the warp barrier orders them
        // before lane 0's copies.
        asm volatile("fence.proxy.async;" ::: "memory");
        __syncwarp();
    }
    uint32_t fwd_phase = 0;           // parity of the transaction being waited for
    bool fwd_inflight = false;        // the last issue_fwd_row started a transaction (warp-uniform)
    auto issue_fwd_row = [&](int y) {            // group A(y)
        const bool have = y >= task.fstart && y >= task.lo;
        if constexpr (TMA_ROWS) {
            fwd_inflight = have;
            if (have && lane == 0)
                bulk_row_to_smem(fwdbuf_a, reinterpret_cast<const char*>(scr) + (long)(y - task.lo) * (128 * PPL), 128 * PPL, fwdbar_a);
        } else {
            if (have) {
                const char* src = reinterpret_cast<const char*>(scr) + (long)(y - task.lo) * (128 * PPL) + lane * (4 * VW);
#pragma unroll
                for (int j = 0; j < PPL / VW; ++j) cp_async8(fwdbuf_lane + j * 256, src + j * 256);
            }
            cp_async_commit();
        }
    };
    auto wait_fwd_row = [&]() {
        if constexpr (TMA_ROWS) {
            if (fwd_inflight) { mbar_wait(fwdbar_a, fwd_phase); fwd_phase ^= 1u; }
        } else {
            cp_async_wait<0>();
        }
    };
    // Depths gathered for an output row stay in registers across the loop back-edge and are stored at the start of
    // the next step: the gather's latency is covered by the row rotation, and nothing else is live meanwhile.
    uint32_t g[NJ * 4];
    auto flush_depth_row = [&](int y) {
        float* pd = out_depth + colbase + (long)y * W;
#pragma unroll
        for (int j = 0; j < NJ; ++j)
            if ((okmask >> j) & 1u) st_stream_v4(pd + j * 128, g[4 * j], g[4 * j + 1], g[4 * j + 2], g[4 * j + 3]);
    };

    issue_fwd_row(task.hi - 1);

    auto bwd_step = [&](const Row<PPL>& A /*row y+1*/, Row<PPL>& Bq /*row y+2 in, row y out*/, int y) {
        if (lane < PPL && y - 3 >= task.fstart)      // forward row three steps ahead -> L2 (one 128 B line per lane)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(scr) +
                                                          (long)(y - 3 - task.lo) * (128 * PPL) + lane * 128));
        if (VEC && y + 1 >= task.r0 && y + 1 < task.r1) flush_depth_row(y + 1);     // gathered during the last step
        wait_fwd_row();                              // A(y), the only transfer in flight, has landed
        uint32_t c[PPL];
        if (y >= task.fstart) {
#pragma unroll
            for (int j = 0; j < PPL / VW; ++j) {
                if (VW == 4) {
                    const uint4 f = reinterpret_cast<const uint4*>(fwdbuf)[j * 32 + lane];
                    c[4 * j] = f.x; c[4 * j + 1] = f.y; c[4 * j + 2] = f.z; c[4 * j + 3] = f.w;
                } else {
                    const uint2 f = fwdbuf[j * 32 + lane];
                    c[2 * j] = f.x; c[2 * j + 1] = f.y;
                }
            }
        } else {
#pragma unroll
            for (int i = 0; i < PPL; ++i) c[i] = init_key;      // rows the forward pass skipped: unreached
        }
#pragma unroll
        for (int i = 0; i < PPL; ++i) c[i] = stencil_bwd<PPL>(c[i], A, Bq, i, fp.one) & ORDCLR;
        if (TMA_ROWS) __syncwarp();                  // every lane has read fwdbuf before the next bulk copy overwrites it
        issue_fwd_row(y - 1);                        // A(y-1): fwdbuf has been consumed above
        constexpr int HF = PPL / 2;                  // chains over columns [HF, PPL) and [0, HF), both right to left
        uint32_t u = c[PPL - 1], u2 = c[HF - 1];
#pragma unroll
        for (int i = 1; i < PPL - HF; ++i) {
            u = __viaddmin_u32(u, KC(1, 1), c[PPL - 1 - i]) & ORDCLR; c[PPL - 1 - i] = u;     // right neighbour is compared last
            if (i < HF) { u2 = __viaddmin_u32(u2, KC(1, 1), c[HF - 1 - i]) & ORDCLR; c[HF - 1 - i] = u2; }
        }
        const uint32_t e = __viaddmin_u32(u | (1u << OSH), uint32_t(HF) << DSH, u2) & ORDCLR;          // lane's first column
        const uint32_t cin = lane_carry<PPL, -1>(e, lane, clamp_dist);
        const uint32_t cin2 = __viaddmin_u32(cin, uint32_t(PPL - HF) << DSH, u) | (1u << OSH);         // column HF, final
#pragma unroll
        for (int i = 0; i < PPL; ++i) {
            uint32_t t = i >= HF ? __viaddmin_u32(cin, uint32_t(PPL - i) << DSH, c[i])
                                 : __viaddmin_u32(cin2, uint32_t(HF - i) << DSH, c[i]);     // order bit 0/1 stays
            if (PAD && x0 + i >= W) t = init_key;
            Bq.v[i] = t;
        }
        refresh_halo(Bq, lane, init_key);

        // ---- output of row y: keys -> shared memory (transpose), then per lane 4 consecutive pixels per group:
        // dt / lbl stores and the gather depth_list[lbl-1] (tools.py:26).  In this layout neighbouring lanes ask
        // for neighbouring labels (consecutive ranks along a beam), so a gather instruction touches few lines.
        // `stage` is re-set every step although it never moves: with `stage_smem` used directly, ptxas orders a few
        // instructions of every instance differently.  This form keeps the SASS that was tuned and measured.
        stage = stage_smem;
        if (y >= task.r0 && y < task.r1) {
#pragma unroll
            for (int j = 0; j < PPL / 2; ++j) swrite[j] = make_uint2(Bq.v[2 * j], Bq.v[2 * j + 1]);
            __syncwarp();
            const long ro = (long)y * W;
            if (VEC) {
                float* pdt = out_dt + colbase + ro;
                int32_t* plb = out_lbl + colbase + ro;
#pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    if ((okmask >> j) & 1u) {
                        const uint4 k = sread[j * 32];
                        if (out_dt)
                            st_stream_v4(pdt + j * 128, __float_as_uint(key_dist_f32(k.x, fp.mul_dist)),
                                         __float_as_uint(key_dist_f32(k.y, fp.mul_dist)),
                                         __float_as_uint(key_dist_f32(k.z, fp.mul_dist)),
                                         __float_as_uint(key_dist_f32(k.w, fp.mul_dist)));
                        if (WANT_LBL)
                            st_stream_v4(plb + j * 128, k.x & LMASK, k.y & LMASK, k.z & LMASK, k.w & LMASK);
                        const uint32_t kk[4] = {k.x, k.y, k.z, k.w};
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const uint32_t l = kk[e] & LMASK;                                // >= 1 inside [c0,c1)
                            g[4 * j + e] = __float_as_uint(*reinterpret_cast<const float*>(dlm1_bytes + (uint64_t)l * fp.four));
                        }
                    }
                }
            } else {
                for (int lc = lane; lc < 32 * PPL; lc += 32) {
                    const int col = task.clo + lc;
                    if (col >= task.c0 && col < task.c1) {
                        const uint32_t k = stage[lc];
                        if (out_dt) out_dt[fpx + ro + col] = (float)(k >> DSH);
                        if (WANT_LBL) out_lbl[fpx + ro + col] = (int32_t)(k & LMASK);
                        out_depth[fpx + ro + col] = dl[(k & LMASK) - 1u];
                    }
                }
            }
            if (y <= task.sky + 1) {                 // base rows S, S+1 of the source-free top rows: keys for k3_sky
                uint32_t* sk = ws.skykeys + ((long)b * 2 + (y - task.sky)) * W;
                for (int lc = lane * 4; lc < 32 * PPL; lc += 128) {
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int col = task.clo + lc + e;
                        if (col >= task.c0 && col < task.c1) sk[col] = stage[lc + e];
                    }
                }
            }
            __syncwarp();                            // stage is free for the next row
        }
    };

#pragma unroll 1
    for (int y = task.hi - 1; y >= task.r0; --y) {
        bwd_step(ra, rb, y);
        const Row<PPL> t = ra; ra = rb; rb = t;
    }
    wait_fwd_row();
    if (VEC) flush_depth_row(task.r0);
}

}  // namespace dtfill
