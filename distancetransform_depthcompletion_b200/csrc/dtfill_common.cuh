// dtfill_common.cuh -- key format, task / parameter / workspace structs and small device helpers shared by the
// kernels of the path (see dtfill_kernels.cuh for the pipeline overview).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace dtfill {


constexpr int DSH = 21;                       // dist field shift
constexpr int OSH = 17;                       // order field shift
constexpr uint32_t LMASK = (1u << OSH) - 1u;  // label field
constexpr uint32_t ORDCLR = ~(15u << OSH);
constexpr uint32_t MAX_FAST_LABEL = LMASK;    // frames with more sources take the wide path
constexpr float UNREACHED_DT = 65533.0f;      // what OpenCV reports where no source is reachable

__host__ __device__ constexpr uint32_t KC(int cost, int order) {
    return (uint32_t(cost) << DSH) | (uint32_t(order) << OSH);
}

// TASK_CHAMFER: full-width tile, the kernel instance with the frame's PPL.  TASK_NARROW: half-width tile, the
// instance with the narrow PPL.  TASK_WIDE: 64-bit-key fallback.  TASK_NOSRC: frame without sources.
enum TaskKind : int { TASK_CHAMFER = 0, TASK_NOSRC = 1, TASK_WIDE = 2, TASK_SKIP = 3, TASK_NARROW = 4 };

// A tile of one frame: the sub-image rows [lo,hi) x columns [clo, clo + 32*PPL) is scanned as if it were the whole
// image; results are written for rows [r0,r1) x columns [c0,c1) only.  Exact because every written pixel's
// city-block ball of radius dt lies inside the sub-image (halo >= a guaranteed bound of dt).
struct __align__(16) Task {
    int frame;
    int lo, hi;        // sub-image rows (band + halo)
    int r0, r1;        // rows whose results are written (lo <= r0 < r1 <= hi)
    int kind;
    int scratch_off;   // start of this task's forward-state scratch, in units of 32 keys
    int fstart;        // first row >= lo holding a source: the forward pass starts here (rows above stay "unreached")
    int clo;           // first column of the sub-image
    int c0, c1;        // columns whose results are written
    int sky;           // S > 0: r0 == S and rows [0,S) of the frame are filled by k3_sky from the final keys of rows
                       // S, S+1, which this task stores into ws.skykeys; -2 otherwise
};

constexpr int MAXT = 32;      // task slots per frame; slot-major layout tasks[slot * B + frame]
constexpr int CELL_H = 4;     // coarse occupancy cells used by the band planner
constexpr int CELL_W = 8;
constexpr int SKY_MAX_W = 1216; // widest frame of the 32-bit-key path (32 lanes x 38 pixels): size of k3_sky's tables
constexpr int MAX_CELLS = 15360;   // planner grid limit (30 KB of shared memory); larger frames are not banded

struct FrameParams {
    int B, H, W, WW;           // WW = 32-bit words per bit row
    int in_H;                  // input frames hold in_H rows
    union {
        int in_crop;           // uint16 input: rows [in_crop, in_crop + H) of an input frame are the frame
        int gt_frames;         // sampled input: frame f of the call reads ground-truth frame f mod gt_frames (several
                               // draws over one ground truth, dtfill_eval_sampled_mt_many; B otherwise)
    };
    float src_thr, val_thr;
    float src_cut;             // smallest float x (in the total order) with !(float32(1 - x) > src_thr)
    int init_dist;             // "unreached" distance of the fast path: H + W + 8
    int force_wide;            // size not representable in the 32-bit key
    int band_cap;              // planner: target cost (row steps) of one task; <= 0 disables banding
    int scratch_units_per_frame; // capacity of the forward-state scratch per frame, in units of 32 keys
    int wide_ppl;              // pixels per lane of the full-width kernel instance (scratch units per row)
    int narrow_ppl;            // pixels per lane of the half-width instance, 0 if frames are never split in columns
    int max_col_tiles;         // planner: at most this many narrow tiles side by side (2..4)
    int sky_min;               // planner: least number of source-free top rows worth handing to k3_sky; 0 disables
    int sky_split;             // planner: the band that feeds k3_sky (rows S..S+3) is a full-width task of its own, so that
                               // k3_sky can follow the full-width launch on the side stream while the narrow tiles still run
    int frame0;                // index of this sub-batch's first frame in the caller's batch (error reporting)
    // Multipliers handed over at run time so that ptxas keeps the multiply-adds below on the FMA pipe instead of
    // strength-reducing them to shifts/LEAs on the ALU pipe, which is the pipe the scan kernel saturates.
    uint32_t mul_dist;         // 1 << (32 - DSH):  umulhi(key, mul_dist)  == key >> DSH
    uint32_t four;             // sizeof(float)
    uint32_t one;              // 1: x * one + c keeps a plain add on the FMA pipe
#ifdef DTFILL_TRACE
    unsigned long long* trace; // tuning build only: per launch {first block start, last block end, sum of block times, blocks}
#endif
};

struct Workspace {
    uint32_t* srcbits;   // [B*H*WW]
    uint16_t* wprefix;   // [B*H*WW] sources in the row before this word
    uint8_t* rowcell;    // [B*H*WW] per word: bit j = some source among its pixels 8j..8j+7
    uint32_t* rowsrc;    // [B*H]  K1: row count, K1b: exclusive base within the frame
    uint32_t* rowval;    // [B*H]
    int32_t* counts;     // [B*2]  n_src, n_valid
    float* dlist;        // [B*H*W] depth_list per frame (first n_valid entries used)
    uint32_t* scratch;   // forward state, lane-major rows of 32*PPL keys
    Task* tasks;         // [B * max_tasks_per_frame]
    int* sky;            // [B] S: rows [0,S) lie above every source and are filled by k3_sky (0: none)
    uint32_t* skykeys;   // [B*2*W] final keys of rows S and S+1
    int* status;         // [0] first bad frame (INT_MAX if none), [1] number of wide tasks
};

// ------------------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float ld_stream(const float* p) {
    float v;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
// Streaming stores to the caller's output buffers: nothing on this path reads them back, so they carry no
// "memory" clobber and the compiler may keep loads in flight across them.
__device__ __forceinline__ void st_stream_u32(void* p, uint32_t v) {
    asm volatile("st.global.cs.u32 [%0], %1;" ::"l"(p), "r"(v));
}
__device__ __forceinline__ void st_stream_v4(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d));
}
// 128-bit read-only load that may allocate in L1: a lane's 16 pixels are four such loads of consecutive 16 B, so
// the second half of every 32 B sector is an L1 hit instead of a second trip to L2
__device__ __forceinline__ float4 ld_stream_v4(const float* p) {
    float4 v;
    asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ uint4 ld_stream_v4u(const void* p) {
    uint4 v;
    asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
// KITTI depth PNG sample -> metres, data_read.py:215 `depth_png.astype(np.float32) / 256.` (exact in float32):
// 0x47000000 is 32768.0f, whose mantissa step is 2^-8, so OR-ing the sample into the mantissa gives 32768 + v/256.
__device__ __forceinline__ float u16_depth(uint32_t v16) { return __uint_as_float(0x47000000u | v16) - 32768.0f; }
__device__ __forceinline__ float load_px_stream(const float* p) { return ld_stream(p); }
__device__ __forceinline__ float load_px_stream(const uint16_t* p) { return u16_depth(__ldg(p)); }

// 16 consecutive pixels of a row as they arrive from memory (128-bit loads), decoded on use
template <typename T> struct In16;
template <> struct In16<float> {
    float4 q[4];
    __device__ __forceinline__ void load(const float* p, int col, int W) {
#pragma unroll
        for (int g = 0; g < 4; ++g) q[g] = col + 4 * g < W ? ld_stream_v4(p + 4 * g) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __device__ __forceinline__ void load_all(const float* p, bool inside) {     // all 16 pixels inside the row, or none
#pragma unroll
        for (int g = 0; g < 4; ++g) q[g] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (inside) {
#pragma unroll
            for (int g = 0; g < 4; ++g) q[g] = ld_stream_v4(p + 4 * g);
        }
    }
    __device__ __forceinline__ float4 get(int g) const { return q[g]; }
};
template <> struct In16<uint16_t> {
    uint4 r[2];
    __device__ __forceinline__ void load(const uint16_t* p, int col, int W) {     // W % 8 == 0
#pragma unroll
        for (int k = 0; k < 2; ++k) r[k] = col + 8 * k < W ? ld_stream_v4u(p + 8 * k) : make_uint4(0u, 0u, 0u, 0u);
    }
    __device__ __forceinline__ void load_all(const uint16_t* p, bool inside) {
        r[0] = r[1] = make_uint4(0u, 0u, 0u, 0u);
        if (inside) { r[0] = ld_stream_v4u(p); r[1] = ld_stream_v4u(p + 8); }
    }
    __device__ __forceinline__ float4 get(int g) const {
        const uint32_t a = (g & 1) ? r[g >> 1].z : r[g >> 1].x, b = (g & 1) ? r[g >> 1].w : r[g >> 1].y;
        return make_float4(u16_depth(a & 0xFFFFu), u16_depth(a >> 16), u16_depth(b & 0xFFFFu), u16_depth(b >> 16));
    }
};
// Input kind of K1 for the NYU loop (dtfill_eval_sampled): dense float32 ground truth, of which only the pixels set in the
// sample bitmap (k10_sample_bits) are kept; the sparse frame `gt * Mask` is formed in registers (dtfill_k1_mask.cuh)
struct SampledGt { float v; };
template <> struct In16<SampledGt> : In16<float> {
    __device__ __forceinline__ void load(const SampledGt* p, int col, int W) { In16<float>::load(&p->v, col, W); }
    __device__ __forceinline__ void load_all(const SampledGt* p, bool inside) { In16<float>::load_all(&p->v, inside); }
};
__device__ __forceinline__ float load_px_stream(const SampledGt* p) { return ld_stream(&p->v); }

// Tuning build (-DDTFILL_TRACE): every block that does work records its start and end (globaltimer, ns) into the
// launch's trace slot, so that the overlap of the kernels of consecutive calls can be reconstructed without a profiler.
#ifdef DTFILL_TRACE
struct TraceScope {
    unsigned long long* t; unsigned long long t0;
    __device__ __forceinline__ TraceScope(const FrameParams& fp, int kernel) : t(fp.trace ? fp.trace + 4 * kernel : nullptr), t0(0) {
        if (t && threadIdx.x == 0) { asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0)); atomicMin(t, t0); }
    }
    __device__ __forceinline__ ~TraceScope() {
        if (t && threadIdx.x == 0) {
            unsigned long long t1; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            atomicMax(t + 1, t1); atomicAdd(t + 2, t1 - t0); atomicAdd(t + 3, 1ull);
        }
    }
};
#define DTFILL_TRACE_SCOPE(fp, k) TraceScope trace_scope_(fp, k)
#else
#define DTFILL_TRACE_SCOPE(fp, k)
#endif

__device__ __forceinline__ uint32_t lanemask_lt() {
    uint32_t m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

}  // namespace dtfill
