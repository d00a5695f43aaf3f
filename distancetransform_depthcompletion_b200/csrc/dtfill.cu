// dtfill.cu -- host side of libdtfill.so: handle, workspace, kernel launches and the C ABI of include/dtfill.h.
#include "dtfill.h"

#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <dlfcn.h>
#include <sched.h>

#include <atomic>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <string>
#include <vector>

#include "dtfill_kernels.cuh"

using namespace dtfill;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

#define CU(call)                                                                                      \
    do {                                                                                              \
        cudaError_t e_ = (call);                                                                      \
        if (e_ != cudaSuccess)                                                                        \
            return fail(DTFILL_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));           \
    } while (0)

struct Buf {
    void* p = nullptr;
    size_t cap = 0;
};

}  // namespace


// ------------------------------------------------------------------------------------------------------------
// Host side of the numpy-in / numpy-out contract (tools.py:13-35 takes and returns ordinary pageable arrays).
// A cudaMemcpyAsync from or to pageable memory is staged by the driver on the calling thread, one chunk at a time,
// and serialises the sliced copy/compute pipeline of dtfill_run.  Pageable buffers are therefore staged here:
// a small pool of threads copies a slice into a pinned mirror (and out of one), the DMA engines move pinned memory
// in both directions, and the kernels of other slices run meanwhile.
// ------------------------------------------------------------------------------------------------------------
// memcpy whose stores bypass the cache (the destination is a staging mirror the CPU does not read back, or the caller's
// array): no read-for-ownership of the destination lines, one third less memory traffic than a plain copy of a buffer
// that does not fit the cache.  Falls back to memcpy on CPUs without AVX2.
#if defined(__x86_64__)
#include <immintrin.h>
__attribute__((target("avx2"))) static void copy_stream_avx2(char* dst, const char* src, size_t n) {
    size_t head = (32 - ((uintptr_t)dst & 31)) & 31;
    if (head > n) head = n;
    if (head) { memcpy(dst, src, head); dst += head; src += head; n -= head; }
    size_t i = 0;
    for (; i + 128 <= n; i += 128) {
        const __m256i a = _mm256_loadu_si256((const __m256i*)(src + i));
        const __m256i b = _mm256_loadu_si256((const __m256i*)(src + i + 32));
        const __m256i c = _mm256_loadu_si256((const __m256i*)(src + i + 64));
        const __m256i d = _mm256_loadu_si256((const __m256i*)(src + i + 96));
        _mm256_stream_si256((__m256i*)(dst + i), a);
        _mm256_stream_si256((__m256i*)(dst + i + 32), b);
        _mm256_stream_si256((__m256i*)(dst + i + 64), c);
        _mm256_stream_si256((__m256i*)(dst + i + 96), d);
    }
    _mm_sfence();
    if (i < n) memcpy(dst + i, src + i, n - i);
}
static void copy_stream(void* dst, const void* src, size_t n) {
    static const bool avx2 = __builtin_cpu_supports("avx2");
    if (avx2 && n >= 4096) copy_stream_avx2((char*)dst, (const char*)src, n);
    else memcpy(dst, src, n);
}
#else
static void copy_stream(void* dst, const void* src, size_t n) { memcpy(dst, src, n); }
#endif

// Sparse upload.  A LiDAR frame is ~95 % pixels that are neither a source (tools.py:8) nor valid (tools.py:22); the path
// never looks at the value of such a pixel, only at the two predicates.  When 0.0f is itself neither (src_cut > 0 and
// val_thr >= 0, true for the reference's thresholds) a pageable input slice is therefore not copied into a pinned mirror
// but compacted by the same host threads into (pixel index, value) pairs of the pixels that satisfy either predicate:
// the threads read the slice once and write ~10 % of it, the link carries 0.4 instead of 4 bytes per pixel, and the
// device rebuilds the dense slice (memset + scatter) in front of K1.  Bit-identical by construction: the predicates are
// evaluated here exactly as K1 evaluates them (NaN is a source), and every dropped pixel is replaced by a value on the
// same side of both.
// A slice's pairs are kept as two arrays: indices [cap], then values [cap].
#if defined(__x86_64__)
struct CompressLut {
    alignas(32) uint32_t perm[256][8];
    CompressLut() {
        for (int m = 0; m < 256; ++m) {
            int k = 0;
            for (int j = 0; j < 8; ++j) if (m & (1 << j)) perm[m][k++] = (uint32_t)j;
            for (; k < 8; ++k) perm[m][k] = 0;
        }
    }
};
// branch-free left-packing: the kept lanes of 8 pixels move to the front with one permute, all 8 lanes are stored and the
// cursor advances by the population count (idx / val need 8 entries of slack)
#define DTFILL_AVX2 __attribute__((target("avx2,popcnt"), always_inline)) static inline
DTFILL_AVX2 __m256 keep8_avx2(const float* p, __m256 vs, __m256 vv) {
    const __m256 x = _mm256_loadu_ps(p);
    return _mm256_or_ps(_mm256_cmp_ps(x, vs, _CMP_NLT_UQ), _mm256_cmp_ps(x, vv, _CMP_GT_OQ));
}
DTFILL_AVX2 size_t emit8_avx2(const CompressLut& lut, const float* p, uint32_t first, unsigned m, uint32_t* idx, uint32_t* val,
                              size_t k) {
    const __m256i iota = _mm256_setr_epi32(0, 1, 2, 3, 4, 5, 6, 7);
    const __m256i perm = _mm256_load_si256((const __m256i*)lut.perm[m]);
    _mm256_storeu_ps((float*)(val + k), _mm256_permutevar8x32_ps(_mm256_loadu_ps(p), perm));
    _mm256_storeu_si256((__m256i*)(idx + k),
                        _mm256_permutevar8x32_epi32(_mm256_add_epi32(_mm256_set1_epi32((int)first), iota), perm));
    return k + (size_t)__builtin_popcount(m);
}
__attribute__((target("avx2,popcnt"))) static size_t compact_block_avx2(const float* src, size_t n, uint32_t base, float scut,
                                                                        float vthr, uint32_t* idx, uint32_t* val) {
    static const CompressLut lut;
    const __m256 vs = _mm256_set1_ps(scut), vv = _mm256_set1_ps(vthr);
    size_t k = 0, i = 0;
    for (; i + 32 <= n; i += 32) {            // most groups of 32 pixels of a LiDAR frame hold nothing: one test
        const __m256 k0 = keep8_avx2(src + i, vs, vv), k1 = keep8_avx2(src + i + 8, vs, vv);
        const __m256 k2 = keep8_avx2(src + i + 16, vs, vv), k3 = keep8_avx2(src + i + 24, vs, vv);
        const __m256 any = _mm256_or_ps(_mm256_or_ps(k0, k1), _mm256_or_ps(k2, k3));
        if (_mm256_testz_ps(any, any)) continue;
        const unsigned m0 = (unsigned)_mm256_movemask_ps(k0), m1 = (unsigned)_mm256_movemask_ps(k1);
        const unsigned m2 = (unsigned)_mm256_movemask_ps(k2), m3 = (unsigned)_mm256_movemask_ps(k3);
        if (m0) k = emit8_avx2(lut, src + i, base + (uint32_t)i, m0, idx, val, k);
        if (m1) k = emit8_avx2(lut, src + i + 8, base + (uint32_t)i + 8, m1, idx, val, k);
        if (m2) k = emit8_avx2(lut, src + i + 16, base + (uint32_t)i + 16, m2, idx, val, k);
        if (m3) k = emit8_avx2(lut, src + i + 24, base + (uint32_t)i + 24, m3, idx, val, k);
    }
    for (; i < n; ++i) {
        const float x = src[i];
        if (!(x < scut) || x > vthr) { memcpy(val + k, &x, 4); idx[k] = base + (uint32_t)i; ++k; }
    }
    return k;
}
// AVX-512: the two predicates of 16 pixels are mask registers, 64 pixels without a hit cost four loads, eight compares and
// one test; the kept lanes are packed by VCOMPRESSPS / VPCOMPRESSD in registers (the register form is fast on every
// AVX-512 core, the memory form is microcoded on some) and all 16 lanes are stored (idx / val need 16 entries of slack)
#define DTFILL_AVX512 __attribute__((target("avx512f,popcnt"), always_inline)) static inline
DTFILL_AVX512 __mmask16 keep16_avx512(const __m512 x, const __m512 vs, const __m512 vv) {
    return (__mmask16)(_mm512_cmp_ps_mask(x, vs, _CMP_NLT_UQ) | _mm512_cmp_ps_mask(x, vv, _CMP_GT_OQ));
}
DTFILL_AVX512 size_t emit16_avx512(const __m512 x, const __mmask16 m, const uint32_t first, uint32_t* idx, uint32_t* val, size_t k) {
    const __m512i iota = _mm512_setr_epi32(0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15);
    _mm512_storeu_ps((float*)(val + k), _mm512_maskz_compress_ps(m, x));
    _mm512_storeu_si512((void*)(idx + k), _mm512_maskz_compress_epi32(m, _mm512_add_epi32(_mm512_set1_epi32((int)first), iota)));
    return k + (size_t)__builtin_popcount((unsigned)m);
}
__attribute__((target("avx512f,popcnt"))) static size_t compact_block_avx512(const float* src, size_t n, uint32_t base, float scut,
                                                                             float vthr, uint32_t* idx, uint32_t* val) {
    const __m512 vs = _mm512_set1_ps(scut), vv = _mm512_set1_ps(vthr);
    size_t k = 0, i = 0;
    for (; i + 64 <= n; i += 64) {
        const __m512 x0 = _mm512_loadu_ps(src + i), x1 = _mm512_loadu_ps(src + i + 16);
        const __m512 x2 = _mm512_loadu_ps(src + i + 32), x3 = _mm512_loadu_ps(src + i + 48);
        const __mmask16 m0 = keep16_avx512(x0, vs, vv), m1 = keep16_avx512(x1, vs, vv);
        const __mmask16 m2 = keep16_avx512(x2, vs, vv), m3 = keep16_avx512(x3, vs, vv);
        if (!((unsigned)m0 | (unsigned)m1 | (unsigned)m2 | (unsigned)m3)) continue;
        if (m0) k = emit16_avx512(x0, m0, base + (uint32_t)i, idx, val, k);
        if (m1) k = emit16_avx512(x1, m1, base + (uint32_t)i + 16, idx, val, k);
        if (m2) k = emit16_avx512(x2, m2, base + (uint32_t)i + 32, idx, val, k);
        if (m3) k = emit16_avx512(x3, m3, base + (uint32_t)i + 48, idx, val, k);
    }
    for (; i + 16 <= n; i += 16) {
        const __m512 x = _mm512_loadu_ps(src + i);
        const __mmask16 m = keep16_avx512(x, vs, vv);
        if (m) k = emit16_avx512(x, m, base + (uint32_t)i, idx, val, k);
    }
    for (; i < n; ++i) {
        const float x = src[i];
        if (!(x < scut) || x > vthr) { memcpy(val + k, &x, 4); idx[k] = base + (uint32_t)i; ++k; }
    }
    return k;
}
#endif
constexpr size_t COMPACT_SLACK = 16;      // entries the packed stores may write beyond the pairs they keep
static size_t compact_block(const float* src, size_t n, uint32_t base, float scut, float vthr, uint32_t* idx, uint32_t* val) {
#if defined(__x86_64__)
    // DTFILL_COMPACT_ISA=avx2|scalar (tuning / tests) keeps the wider paths off
    static const int isa = [] {
        const char* e = getenv("DTFILL_COMPACT_ISA");
        const int limit = !e ? 3 : (!strcmp(e, "scalar") ? 0 : (!strcmp(e, "avx2") ? 2 : 3));
        if (limit >= 3 && __builtin_cpu_supports("avx512f") && __builtin_cpu_supports("popcnt")) return 3;
        if (limit >= 2 && __builtin_cpu_supports("avx2") && __builtin_cpu_supports("popcnt")) return 2;
        return 0;
    }();
    if (isa == 3) return compact_block_avx512(src, n, base, scut, vthr, idx, val);
    if (isa == 2) return compact_block_avx2(src, n, base, scut, vthr, idx, val);
#endif
    size_t k = 0;
    for (size_t i = 0; i < n; ++i) {
        const float x = src[i];
        if (!(x < scut) || x > vthr) { memcpy(val + k, &x, 4); idx[k] = base + (uint32_t)i; ++k; }
    }
    return k;
}

class CopyPool {
public:
    explicit CopyPool(int n) {
        for (int i = 0; i < n; ++i) th_.emplace_back([this] { loop(); });
    }
    ~CopyPool() {
        { std::lock_guard<std::mutex> lk(mu_); stop_ = true; }
        cv_.notify_all();
        for (auto& t : th_) t.join();
    }
    // fn(0) .. fn(nparts - 1), split over the pool's threads and the caller; returns when all are done
    void parallel_for(size_t nparts, const std::function<void(size_t)>& fn) {
        if (nparts <= 1 || th_.empty()) { for (size_t i = 0; i < nparts; ++i) fn(i); return; }
        {
            std::lock_guard<std::mutex> lk(mu_);
            fn_ = &fn; nparts_ = nparts; next_ = 0; done_ = 0;
        }
        cv_.notify_all();
        work();
        std::unique_lock<std::mutex> lk(mu_);
        cv_done_.wait(lk, [this] { return done_ == nparts_; });
        nparts_ = 0;
    }
    // dst[0..bytes) = src[0..bytes)
    void copy(void* dst, const void* src, size_t bytes) {
        const size_t grain = 2u << 20;
        const size_t nparts = bytes / grain > 0 ? std::min<size_t>(bytes / grain, (th_.size() + 1) * 4) : 1;
        parallel_for(nparts, [=](size_t i) {
            const size_t a = bytes * i / nparts, b = bytes * (i + 1) / nparts;
            copy_stream((char*)dst + a, (const char*)src + a, b - a);
        });
    }
    // indices and values of the pixels of src[0..n) that are a source or valid -> idx[0..count), val[0..count); returns
    // count, or SIZE_MAX if they do not fit into cap entries (the caller then copies the slice densely)
    size_t compact(uint32_t* idx, uint32_t* val, size_t cap, const float* src, size_t n, float scut, float vthr) {
        const size_t block = 1u << 15;                       // pixels per work item
        const size_t nparts = (n + block - 1) / block;
        std::atomic<size_t> cursor{0};
        std::atomic<bool> overflow{false};
        parallel_for(nparts, [&](size_t i) {
            if (overflow.load(std::memory_order_relaxed)) return;
            thread_local std::vector<uint32_t> buf;
            if (buf.size() < 2 * (block + COMPACT_SLACK)) buf.resize(2 * (block + COMPACT_SLACK));
            uint32_t* bi = buf.data();
            uint32_t* bv = buf.data() + block + COMPACT_SLACK;
            const size_t a = i * block, len = std::min(block, n - a);
            const size_t k = compact_block(src + a, len, (uint32_t)a, scut, vthr, bi, bv);
            const size_t off = cursor.fetch_add(k);
            if (off + k > cap) { overflow.store(true); return; }
            memcpy(idx + off, bi, k * 4);
            memcpy(val + off, bv, k * 4);
        });
        return overflow.load() ? SIZE_MAX : cursor.load();
    }

private:
    void work() {
        for (;;) {
            size_t i;
            const std::function<void(size_t)>* fn;
            {
                std::lock_guard<std::mutex> lk(mu_);
                if (next_ >= nparts_) return;
                i = next_++;
                fn = fn_;
            }
            (*fn)(i);
            std::lock_guard<std::mutex> lk(mu_);
            if (++done_ == nparts_) cv_done_.notify_all();
        }
    }
    void loop() {
        for (;;) {
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [this] { return stop_ || next_ < nparts_; });
                if (stop_) return;
            }
            work();
        }
    }
    std::vector<std::thread> th_;
    std::mutex mu_;
    std::condition_variable cv_, cv_done_;
    bool stop_ = false;
    const std::function<void(size_t)>* fn_ = nullptr;
    size_t nparts_ = 0, next_ = 0, done_ = 0;
};

struct PinBuf {
    void* p = nullptr;
    size_t cap = 0;
};

// One "lane" = everything a call needs while it is in flight: workspace, streams, events.  A handle has two, so
// that in pipelined mode (dtfill_set_pipeline_depth 2) the HBM-bound first stage of one call overlaps the ALU-bound
// scan of the previous call.
struct Lane {
    static const int MAX_SUB = 16;
    Buf srcbits, wprefix, rowcell, rowsrc, rowval, counts, dlist, scratch, tasks, sky, skykeys;
    Buf ev_partial, ev_per_frame, ev_totals;   // dtfill_run_eval_async: metric partial sums / per-frame metrics / running totals
    bool ev_dirty = false;                     // ev_totals holds sums not yet collected by dtfill_eval_totals
    cudaStream_t sub[MAX_SUB] = {};      // sub-batch streams (host buffers: slices pipeline the PCIe copies)
    cudaEvent_t fork_ev = nullptr, join_ev[MAX_SUB] = {};
    cudaStream_t side[MAX_SUB] = {};     // narrow tiles run next to the full-width tasks of the same sub-batch
    cudaEvent_t side_fork[MAX_SUB] = {}, side_join[MAX_SUB] = {};
    cudaStream_t pipe = nullptr;         // pipelined mode: the stream this lane's calls run on
    cudaEvent_t done = nullptr;          // ... and the end of its last call
    bool pending = false;                // done not yet waited for by the handle's stream
    int last_launches = 0;
    int last_B = 0;
};

struct dtfill_ctx {
    int device = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    int sm_count = 148;
    static const int MAX_LANES = 4;      // measured with 8: depth 5 0.416, 6 0.434, 8 0.470 ms per step against 0.413 at 4
    Lane lanes[MAX_LANES];
    int ncalls = 0;                   // calls enqueued so far (pipelined mode alternates lanes)
    int last_lane = 0;
    // Outcome of every call since the last dtfill_status: call n copies its two status words (first bad frame, wide
    // tasks) into slot n % STATUS_RING of a pinned ring that only the device writes after the host armed it, so no call's
    // IndexError can be overwritten by a later call.  A slot still unexamined when the ring wraps is folded into
    // `sticky_bad` after waiting for its call.
    static const int STATUS_RING = 64;
    int* status_ring = nullptr;       // pinned [STATUS_RING][2]
    int* status_init = nullptr;       // pinned {INT_MAX, 0}: what every call's device status words start from
    bool slot_dirty[STATUS_RING] = {};
    cudaEvent_t slot_done[STATUS_RING] = {};
    int sticky_bad = INT_MAX;
    // The device side of a slot: STATUS_STRIDE ints per slot in one allocation, {INT_MAX, 0, ...} from dtfill_create on.
    // A call's kernels only ever change them for a bad frame or a 64-bit-key frame, so a slot whose host copy came back
    // unchanged needs no re-arming before its next use, and the copy to the host is issued right behind
    // k1b_scan_compact (the only writer) on a stream of its own: neither transfer sits between two calls' kernels
    // (they cost ~8 us per call: one KITTI frame 0.135 -> see profiles/r02_experiments.txt).
    static const int STATUS_STRIDE = 64;
    int* status_dev = nullptr;        // device [STATUS_RING][STATUS_STRIDE]
    bool slot_rearm[STATUS_RING] = {}; // the slot's device words left their initial state: re-arm before the next use
    cudaStream_t status_stream = nullptr;
    cudaEvent_t status_fork = nullptr;
    int* cur_status = nullptr;        // device status words of the call being enqueued
    int cur_slot = 0;
    bool cur_status_early = false;    // this call copies its status words to the host right behind k1b_scan_compact
    bool cur_status_copied = false;
    int last_slot = 0;
    std::vector<void*> retired;       // device buffers replaced by larger ones; freed at the next synchronisation point
    size_t wide_smem_configured = 0;  // dynamic shared memory limit of k2_chamfer_wide raised so far on this device
    bool cur_pipelined = false;       // the call being enqueued runs on a lane's own stream
    // input of the call being enqueued: float32 frames [B,H,W], or uint16 PNG samples [B,in_H,W] of which rows
    // [in_crop, in_crop + H) are the frame (dtfill_run_u16); lidar_dev: decoded float32 frames, optional
    bool in_u16 = false;
    int in_H = 0, in_crop = 0;
    float* lidar_dev = nullptr;
    // ... or dense float32 ground truth [B,H,W] of which K1 keeps the pixels of the sample bitmap that k10_sample_bits left
    // in lane 0's srcbits (dtfill_eval_sampled)
    bool in_sampled = false;
    // evaluation fused behind the call being enqueued (dtfill_run_eval_async): ground truth, mode
    const void* ev_gt = nullptr;
    int ev_gt_f64 = 0, ev_mode = 0;
    int pipeline_depth = 1;           // 1: strict stream order (default); 2: consecutive calls may overlap
    cudaEvent_t pipe_fork = nullptr;
    Buf in_dev, depth_dev, dt_dev, lbl_dev, mask_dev, counts_out_dev, lidar_out_dev;   // staging for host-pointer calls
    Buf gt_dev, partial, per_frame, sums, edt_rows, edt_stack;
    // pinned mirrors of pageable caller buffers (see CopyPool) and the threads that fill / drain them
    PinBuf pin_in, pin_depth, pin_dt, pin_lbl, pin_mask, pin_lidar, pin_sparse;
    Buf sparse_dev;                   // (index, value) pairs of a sparse upload, per slice
    Buf mx_terms, mx_counts, mx_leaf_start, mx_leaf_sum;     // dtfill_metrics in numpy's summation order (k4x_*)
    // PNG decode (k8_png_*): uploaded files + offsets, filtered bytes per frame, decoded samples (dtfill_run_png), status
    Buf png_data, png_scratch, png_samples, png_status;
    PinBuf pin_png, pin_png_status;   // pinned staging of host file bytes / of the per-frame status
    // PNG encode (k9_png_*): uploaded input, filtered bytes, row Adler-32s, segment chunks and sizes, packed files and
    // their offsets (host outputs), filled depth of dtfill_run_png_to_png
    Buf enc_in, enc_filt, enc_adler, enc_slots, enc_seg, enc_out, enc_off, enc_depth;
    PinBuf pin_enc_off;
    // dtfill_eval_sampled: uploaded host coordinates, the flag word of k10_sample_bits; pinned staging of host coordinates,
    // and of the counts and the flag word on their way back
    Buf smp_coords, smp_bad;
    PinBuf pin_smp, pin_smp_out;
    bool metrics_exact = true;        // dtfill_metrics / _ex reproduce np.mean's pairwise sums bit for bit
    bool sparse_upload = true;        // pageable float32 inputs are compacted on the host instead of mirrored (see CopyPool)
    size_t last_h2d_bytes = 0, last_d2h_bytes = 0;   // bytes the last synchronous host call moved over the link
    CopyPool* pool_in = nullptr;
    CopyPool* pool_out = nullptr;
    int stage_threads = -1;           // threads per direction; -1: automatic; 0: never stage (driver-staged copies)
    int32_t* counts_host = nullptr;   // pinned staging for out_counts (a pageable destination would serialise the
    size_t counts_host_cap = 0;       // sliced copies: cudaMemcpyAsync to pageable memory blocks the host)
    bool profiling = false;
#ifdef DTFILL_TRACE
    unsigned long long* trace_dev = nullptr;   // [TRACE_CALLS][4 kernels][4]
    static const int TRACE_CALLS = 256;
#endif
    int debug_skip = 0;               // tuning only (dtfill_debug_set_skip): bit 0 K1, 1 K1b, 2 K2, 3 k3_sky are not launched
    int sky_min = -1;             // source-free top rows go to k3_sky when there are at least this many; 0: never;
                                  // -1: automatic = 8 (measured in strict order on KITTI-64 frames: one frame 0.209 ->
                                  // 0.137 ms, 16 frames 0.222 -> 0.165, 256 frames 0.551 -> 0.536; the launch costs
                                  // 2 % on frames without such rows, 256 NYU frames 0.603 -> 0.616)
    int nsub = -1;                // -1: automatic
    int band_cap = -1;            // -1: automatic (see enqueue); 0: never split frames; >0: task cost target in row steps
    cudaEvent_t ev[DTFILL_NUM_KERNELS + 1] = {};
};

namespace {

int ensure(dtfill_t* h, Buf& b, size_t bytes) {
    if (bytes <= b.cap) return 0;
    if (b.p) {
        // work in flight may still use the old buffer: park it, dtfill_synchronize / dtfill_destroy free it
        h->retired.push_back(b.p);
        b.p = nullptr;
        b.cap = 0;
    }
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) {
        b.p = nullptr;
        return fail(DTFILL_E_NOMEM, std::string("cudaMalloc(") + std::to_string(want) + "): " + cudaGetErrorString(e));
    }
    b.cap = want;
    return 0;
}

// Host buffers of a dtfill_run call with host pointers: each sub-batch copies its own slices on its own stream, so
// the host->device copy of one slice, the kernels of another and the device->host copy of a third overlap.
struct HostIO {
    const void* in = nullptr;
    float* lidar = nullptr;
    float* depth = nullptr;
    float* dt = nullptr;
    int32_t* lbl = nullptr;
    uint8_t* mask = nullptr;
    int32_t* counts = nullptr;
    // pinned mirrors for the buffers above that are pageable (nullptr: the caller's buffer is pinned, copy directly)
    void* in_pin = nullptr;
    float* lidar_pin = nullptr;
    float* depth_pin = nullptr;
    float* dt_pin = nullptr;
    int32_t* lbl_pin = nullptr;
    uint8_t* mask_pin = nullptr;
    bool any_out_pin() const { return lidar_pin || depth_pin || dt_pin || lbl_pin || mask_pin; }
    // sparse upload of a pageable float32 input (instead of in_pin): pinned pair buffer, pairs per pixel it can hold
    uint32_t* sparse_pin = nullptr;   // per slice: indices [cap], values [cap]
    size_t sparse_cap_div = 0;        // capacity of a slice of n pixels: cap = n / sparse_cap_div pairs
    float sparse_scut = 0.f, sparse_vthr = 0.f;
};

bool is_pageable(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return a.type == cudaMemoryTypeUnregistered;
}

int ensure_pinned(PinBuf& b, size_t bytes) {
    if (bytes <= b.cap) return 0;
    if (b.p) { cudaFreeHost(b.p); b.p = nullptr; b.cap = 0; }
    const size_t want = bytes + bytes / 16 + 4096;
    cudaError_t e = cudaHostAlloc(&b.p, want, cudaHostAllocDefault);
    if (e != cudaSuccess) { b.p = nullptr; return fail(DTFILL_E_NOMEM, std::string("cudaHostAlloc(") + std::to_string(want) + "): " + cudaGetErrorString(e)); }
    b.cap = want;
    return 0;
}

// dense slice = zeros + the pairs of a sparse upload (see CopyPool::compact)
__global__ void __launch_bounds__(256) k0_scatter_pairs(const uint32_t* __restrict__ idx, const uint32_t* __restrict__ val,
                                                         unsigned n, float* __restrict__ dst)
{
    const unsigned i = blockIdx.x * 256u + threadIdx.x;
    if (i < n) dst[idx[i]] = __uint_as_float(val[i]);
}

struct Plan {
    int ppl = 0;        // pixels per lane of the full-width instance; 0: 64-bit-key path only
    bool pad = false;
    int wp = 0;         // padded row width of the scratch
    int narrow = 0;     // pixels per lane of the half-width instance (two overlapping tiles per band), 0: none
};

Plan make_plan(int H, int W) {
    Plan p;
    const int cand[3] = {10, 20, 38};
    for (int c : cand) {
        if (W <= 32 * c && 2 * H + W + c + 12 <= 2047) {
            p.ppl = c;
            p.pad = (W != 32 * c);
            p.wp = 32 * c;
            // half-width tiles need an overlap: two tiles of 32*narrow columns must cover W with room for halos
            if (c == 38 && W > 640 + 16 && (W & 3) == 0) p.narrow = 20;
            if (c == 20 && W > 320 + 16 && W <= 640 - 48 && (W & 3) == 0) p.narrow = 10;
            return p;
        }
    }
    p.ppl = 0;
    p.wp = W;
    return p;
}

template <int PPL, bool PAD, bool LBL>
void launch_k2b(bool vec, int grid, cudaStream_t s, const FrameParams& fp, const Workspace& ws, float* od, float* odt,
                int32_t* ol, int kind) {
    if (vec) k2_chamfer<PPL, PAD, LBL, true><<<grid, 32, 0, s>>>(fp, ws, od, odt, ol, kind);
    else k2_chamfer<PPL, PAD, LBL, false><<<grid, 32, 0, s>>>(fp, ws, od, odt, ol, kind);
}

template <int PPL>
void launch_k2(bool pad, bool want_lbl, int grid, cudaStream_t s, const FrameParams& fp, const Workspace& ws,
               float* od, float* odt, int32_t* ol, int kind) {
    const bool vec = (fp.W & 3) == 0;      // row starts 16-byte aligned: 128-bit output stores
    if (pad) {
        if (want_lbl) launch_k2b<PPL, true, true>(vec, grid, s, fp, ws, od, odt, ol, kind);
        else launch_k2b<PPL, true, false>(vec, grid, s, fp, ws, od, odt, ol, kind);
    } else {
        if (want_lbl) launch_k2b<PPL, false, true>(vec, grid, s, fp, ws, od, odt, ol, kind);
        else launch_k2b<PPL, false, false>(vec, grid, s, fp, ws, od, odt, ol, kind);
    }
}

// tools.py:8 marks a pixel as source when !(float32(1 - x) > src_thr).  The predicate is monotone in x (false below,
// true above; NaN inputs are sources), so it equals !(x < cut) for the smallest float `cut` that satisfies it.
// Bisection over the floats in their total order (-inf .. -0 < +0 .. +inf); K1 then needs one subtraction per pixel.
static inline float ordered_to_float(uint32_t k) {
    const uint32_t b = (k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k;
    float f; memcpy(&f, &b, 4); return f;
}
static float source_cut(float thr) {
    auto is_src = [thr](float x) { volatile float d = 1.0f - x; return !(d > thr); };
    uint32_t lo = 0x007FFFFFu, hi = 0xFF800000u;      // ordered keys of -inf and +inf; is_src(+inf) always holds
    if (is_src(ordered_to_float(lo))) return ordered_to_float(lo);
    while (hi - lo > 1) {                             // invariant: !is_src(lo), is_src(hi)
        const uint32_t mid = lo + (hi - lo) / 2;
        if (is_src(ordered_to_float(mid))) hi = mid; else lo = mid;
    }
    return ordered_to_float(hi);
}

constexpr int MAX_COL_TILES = 4;      // planner: at most this many half-width tiles side by side in a band

// Enqueue the path for frames [b0, b0+nb) of the batch on stream s; all pointers are device pointers to the whole
// batch, the workspace is sliced per frame so sub-batches never share anything but the status words.
int enqueue_range(dtfill_t* h, Lane* L, cudaStream_t s, const Plan& plan, int b0, int nb, int Btot, const void* in, int H, int W,
                  float src_thr, float val_thr, float* out_depth, float* out_dt, int32_t* out_lbl, uint8_t* out_mask,
                  int32_t* out_counts, int scratch_units_per_frame, int sub_index, int* launches) {
    const int WW = (W + 31) / 32;
    const size_t rows0 = (size_t)b0 * H, npx0 = rows0 * W;
    const size_t rows = (size_t)nb * H;
    FrameParams fp;
    fp.B = nb; fp.H = H; fp.W = W; fp.WW = WW;
    fp.in_H = h->in_u16 ? h->in_H : H;
    fp.in_crop = h->in_u16 ? h->in_crop : 0;
    fp.src_thr = src_thr; fp.val_thr = val_thr;
    fp.src_cut = source_cut(src_thr);
    fp.init_dist = H + W + 8;
    fp.force_wide = plan.ppl == 0;
    fp.scratch_units_per_frame = scratch_units_per_frame;
    fp.wide_ppl = plan.ppl ? plan.ppl : 1;
    fp.narrow_ppl = plan.ppl ? plan.narrow : 0;
    fp.frame0 = b0;
    fp.sky_min = h->sky_min >= 0 ? h->sky_min : 8;
    // strict order with two scan instances: k3_sky follows the full-width instance on the side stream (see the planner)
    // -- while the scan leaves SMs idle: measured on KITTI frames, 4 / 16 / 32 / 64 frames per call -4 / -10 / -9 / -2 %,
    // 128 / 256 frames +4 / +2 % (the wide instance then takes registers from the narrow tiles)
    fp.sky_split = (!h->cur_pipelined && !h->profiling && plan.ppl && plan.narrow && fp.sky_min > 0 && W <= SKY_MAX_W &&
                    (long)Btot * H * W <= 28000000L) ? 1 : 0;
    fp.max_col_tiles = MAX_COL_TILES;
    fp.mul_dist = 1u << (32 - DSH);
    fp.four = 4u;
    fp.one = 1u;
#ifdef DTFILL_TRACE
    fp.trace = h->trace_dev ? h->trace_dev + (size_t)(h->ncalls % dtfill_ctx::TRACE_CALLS) * 16 : nullptr;
#endif
    {   // band planner target: enough independent tiles to keep ~24 warps per SM busy over the whole batch
        int cap = h->band_cap;
        if (cap < 0) {
            // tiles wanted per frame; with batches overlapping (pipelined mode) fewer, taller tiles do: they carry
            // less halo redundancy and the other batches in flight fill the SMs
            // (measured on 256 KITTI frames, 4 batches in flight: target 260 -> 0.417 ms per step, 202 -> 0.426, 330 -> 0.419)
            const long beff = h->pipeline_depth > 1 ? (9L * Btot + 3) / 4 : Btot;
            const long per_frame = ((long)h->sm_count * 28 + beff - 1) / beff;
            if (per_frame <= 1) cap = 0;                                              // batch alone fills the GPU
            else {
                const long band_rows = (5L * H / 2) / per_frame;                       // ~2.5 tiles per band of rows
                cap = (int)(2 * band_rows + 42);
                // (the floor: bands shorter than twice their halo are not cut anyway; measured on KITTI frames, 1 / 4 frames
                // per call 0.129 -> 0.119 / 0.133 -> 0.126 ms with 80 instead of 96, 16 frames 0.144 -> 0.150)
                const int floor_cap = Btot <= 8 ? 80 : 96;
                if (cap < floor_cap) cap = floor_cap;
            }
        }
        fp.band_cap = plan.ppl ? cap : 0;
    }
    Workspace ws;
    ws.srcbits = (uint32_t*)L->srcbits.p + rows0 * WW;
    ws.wprefix = (uint16_t*)L->wprefix.p + rows0 * WW;
    ws.rowcell = (uint8_t*)L->rowcell.p + rows0 * WW;
    ws.rowsrc = (uint32_t*)L->rowsrc.p + rows0;
    ws.rowval = (uint32_t*)L->rowval.p + rows0;
    ws.counts = (int32_t*)L->counts.p + 2 * (size_t)b0;
    ws.dlist = (float*)L->dlist.p + npx0;
    ws.scratch = (uint32_t*)L->scratch.p + (size_t)b0 * scratch_units_per_frame * 32;
    ws.tasks = (Task*)L->tasks.p + (size_t)b0 * MAXT;
    ws.status = h->cur_status;
    ws.sky = (int*)L->sky.p + b0;
    ws.skykeys = (uint32_t*)L->skykeys.p + (size_t)b0 * 2 * W;
    float* olid = h->lidar_dev ? h->lidar_dev + npx0 : nullptr;
    float* od = out_depth + npx0;
    float* odt = out_dt ? out_dt + npx0 : nullptr;
    int32_t* ol = out_lbl ? out_lbl + npx0 : nullptr;
    uint8_t* om = out_mask ? out_mask + npx0 : nullptr;
    int32_t* oc = out_counts ? out_counts + 2 * (size_t)b0 : nullptr;

    if (h->profiling) CU(cudaEventRecord(h->ev[0], s));
    if (!(h->debug_skip & 1)) {   // K1: one warp per row
        // small blocks (2 warps, no shared memory): they fit into the registers the scan's warps of other batches
        // leave free on an SM, so K1 starts flowing before those drain (measured: 256 -> 64 threads, step -2 %)
        const int k1_threads = 64;
        const int wpb = k1_threads / 32;
        long want = ((long)rows + wpb - 1) / wpb;
        int grid = (int)(want < 1 ? 1 : want);
        if (h->in_sampled) {
            const SampledGt* in_s = (const SampledGt*)in + npx0;
            if ((W & 15) == 0) k1_mask_rows_v16<SampledGt, true><<<grid, k1_threads, 0, s>>>(in_s, fp, ws, om, olid);
            else if ((W & 3) == 0) k1_mask_rows_v16<SampledGt, false><<<grid, k1_threads, 0, s>>>(in_s, fp, ws, om, olid);
            else k1_mask_rows<SampledGt><<<grid, k1_threads, 0, s>>>(in_s, fp, ws, om, olid);
        } else if (!h->in_u16) {
            const float* in_s = (const float*)in + npx0;
            if ((W & 15) == 0) k1_mask_rows_v16<float, true><<<grid, k1_threads, 0, s>>>(in_s, fp, ws, om, nullptr);
            else if ((W & 3) == 0) k1_mask_rows_v16<float, false><<<grid, k1_threads, 0, s>>>(in_s, fp, ws, om, nullptr);
            else k1_mask_rows<float><<<grid, k1_threads, 0, s>>>(in_s, fp, ws, om, nullptr);
        } else {
            const uint16_t* in_s = (const uint16_t*)in + (size_t)b0 * h->in_H * W;
            if ((W & 15) == 0) k1_mask_rows_v16<uint16_t, true><<<grid, k1_threads, 0, s>>>(in_s, fp, ws, om, olid);
            else if ((W & 7) == 0) k1_mask_rows_v16<uint16_t, false><<<grid, k1_threads, 0, s>>>(in_s, fp, ws, om, olid);
            else k1_mask_rows<uint16_t><<<grid, k1_threads, 0, s>>>(in_s, fp, ws, om, olid);
        }
        ++*launches;
    }
    if (h->profiling) CU(cudaEventRecord(h->ev[1], s));
    if (!(h->debug_skip & 2)) {
        k1b_scan_compact<<<nb, K1B_THREADS, 0, s>>>(fp, ws, oc);
        ++*launches;
        if (h->cur_status_early) {       // the status words are final: to the host on the status stream
            CU(cudaEventRecord(h->status_fork, s));
            CU(cudaStreamWaitEvent(h->status_stream, h->status_fork, 0));
            CU(cudaMemcpyAsync(h->status_ring + 2 * h->cur_slot, h->cur_status, 8, cudaMemcpyDeviceToHost, h->status_stream));
            CU(cudaEventRecord(h->slot_done[h->cur_slot], h->status_stream));
            h->cur_status_copied = true;
        }
    }
    if (h->profiling) CU(cudaEventRecord(h->ev[2], s));

    const bool want_lbl = ol != nullptr;
    // half-width and full-width tiles are different kernel instances and run next to each other on two streams.  The
    // instance that a frame of this shape normally uses stays on the call's own stream, so that the chain
    // K1 -> K1b -> scan -> k3_sky does not cross streams twice (narrow_main; the other instance finds no task as a rule;
    // measured with the instances the other way round: strict step of 256 KITTI frames 0.536 ms against 0.519)
    const bool run_k2 = !(h->debug_skip & 4);
    const bool two = fp.narrow_ppl && run_k2;
    const bool narrow_main = two && !h->profiling;
    cudaStream_t s_side = s;
    if (two) {
        s_side = L->side[sub_index];
        CU(cudaEventRecord(L->side_fork[sub_index], s));
        CU(cudaStreamWaitEvent(s_side, L->side_fork[sub_index], 0));
    }
    cudaStream_t s_narrow = narrow_main ? s : s_side, s_full = narrow_main ? s_side : s;
    if (two) {
        if (fp.narrow_ppl == 20) launch_k2<20>(false, want_lbl, nb * MAXT, s_narrow, fp, ws, od, odt, ol, TASK_NARROW);
        else launch_k2<10>(false, want_lbl, nb * MAXT, s_narrow, fp, ws, od, odt, ol, TASK_NARROW);
        ++*launches;
    }
    if (run_k2) switch (plan.ppl) {
        case 10: launch_k2<10>(plan.pad, want_lbl, nb * MAXT, s_full, fp, ws, od, odt, ol, TASK_CHAMFER); break;
        case 20: launch_k2<20>(plan.pad, want_lbl, nb * MAXT, s_full, fp, ws, od, odt, ol, TASK_CHAMFER); break;
        case 38: launch_k2<38>(plan.pad, want_lbl, nb * MAXT, s_full, fp, ws, od, odt, ol, TASK_CHAMFER); break;
        default: launch_k2<10>(true, want_lbl, nb * MAXT, s_full, fp, ws, od, odt, ol, TASK_CHAMFER); break;  // NOSRC only
    }
    if (run_k2) ++*launches;
    // 64-bit-key fallback: returns immediately for every task the fast kernels handle.  It touches other frames
    // than they do, so it runs next to the narrow tiles; only per-kernel profiling serialises it behind the join.
    const size_t wide_smem = (size_t)3 * (W + 4) * sizeof(uint64_t);
    if (!h->profiling && run_k2) {
        k2_chamfer_wide<<<nb, 32, wide_smem, s_full>>>(fp, ws, od, odt, ol);
        ++*launches;
    }
    const bool run_sky = fp.band_cap > 0 && fp.sky_min > 0 && W <= SKY_MAX_W && !(h->debug_skip & 8);
    bool sky_done = false;
    if (two && narrow_main && fp.sky_split && run_sky) {
        // the base rows of every frame come from the full-width instance just launched on the side stream
        k3_sky<<<dim3(nb, (H + SKY_ROWS - 1) / SKY_ROWS), 256, 0, s_side>>>(fp, ws, od, odt, ol);
        ++*launches;
        sky_done = true;
    }
    if (two) {
        CU(cudaEventRecord(L->side_join[sub_index], s_side));
        CU(cudaStreamWaitEvent(s, L->side_join[sub_index], 0));
    }
    if (h->profiling) {
        CU(cudaEventRecord(h->ev[3], s));
        k2_chamfer_wide<<<nb, 32, wide_smem, s>>>(fp, ws, od, odt, ol);
        ++*launches;
        CU(cudaEventRecord(h->ev[4], s));
    }
    // rows above the first source row, from the two base rows the scan left in ws.skykeys (blocks of frames without
    // such rows return at once)
    if (run_sky && !sky_done) {
        k3_sky<<<dim3(nb, (H + SKY_ROWS - 1) / SKY_ROWS), 256, 0, s>>>(fp, ws, od, odt, ol);
        ++*launches;
    }
    if (h->profiling) CU(cudaEventRecord(h->ev[5], s));
    return 0;
}

// Enqueue the whole path on h->stream; all pointers are device pointers.
int enqueue(dtfill_t* h, const void* in, int B, int H, int W, float src_thr, float val_thr, float* out_depth,
            float* out_dt, int32_t* out_lbl, uint8_t* out_mask, int32_t* out_counts, const HostIO* hio = nullptr,
            bool force_strict = false) {
    if (!h || !in || !out_depth) return fail(DTFILL_E_ARG, "dtfill_run: NULL handle, input or out_depth");
    if (B <= 0 || H <= 0 || W <= 0) return fail(DTFILL_E_ARG, "dtfill_run: B, H, W must be positive");
    if ((long)H + W >= 60000 || (long)H * W >= (1l << 31) || W > 28000)
        return fail(DTFILL_E_ARG, "dtfill_run: frame size not supported (H + W < 60000, W <= 28000)");
    CU(cudaSetDevice(h->device));
    // lane and stream of this call
    // synchronous entries (dtfill_run*) always run in strict order on the handle's stream: their device-to-host copies
    // and their status follow the kernels in stream order
    const bool pipelined = h->pipeline_depth > 1 && !h->profiling && !hio && !force_strict;
    Lane* L = &h->lanes[pipelined ? (h->ncalls % h->pipeline_depth) : 0];
    h->cur_pipelined = pipelined;
    const Plan plan = make_plan(H, W);
    const int WW = (W + 31) / 32;
    const size_t rows = (size_t)B * H;
    const size_t npx = rows * W;

    int rc;
    if ((rc = ensure(h, L->srcbits, rows * WW * 4))) return rc;
    if ((rc = ensure(h, L->wprefix, rows * WW * 2))) return rc;
    if ((rc = ensure(h, L->rowcell, rows * WW))) return rc;
    if ((rc = ensure(h, L->rowsrc, rows * 4))) return rc;
    if ((rc = ensure(h, L->rowval, rows * 4))) return rc;
    if ((rc = ensure(h, L->counts, (size_t)B * 8))) return rc;
    if ((rc = ensure(h, L->dlist, npx * 4))) return rc;
    // forward-state scratch in units of 32 keys: tiles overlap by their halos, so allow 3 H full-width rows per
    // frame (the 64-bit-key path keeps one u32 per pixel there; K1 parks H*W floats there as well)
    const int scratch_units_per_frame = plan.ppl ? 3 * H * plan.ppl : (int)(((size_t)H * W + 31) / 32);
    if ((rc = ensure(h, L->scratch, (size_t)B * scratch_units_per_frame * 128))) return rc;
    if ((rc = ensure(h, L->tasks, (size_t)B * MAXT * sizeof(Task)))) return rc;
    if ((rc = ensure(h, L->sky, (size_t)B * 4))) return rc;
    if ((rc = ensure(h, L->skykeys, (size_t)B * 2 * W * 4))) return rc;
    {
        const size_t smem = (size_t)3 * (W + 4) * sizeof(uint64_t);
        if (smem > 227 * 1024) return fail(DTFILL_E_ARG, "dtfill_run: frame too wide for the wide path");
        if (smem > 48 * 1024 && smem > h->wide_smem_configured) {     // the attribute is per device: track it per handle
            CU(cudaFuncSetAttribute(k2_chamfer_wide, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            h->wide_smem_configured = smem;
        }
    }

    cudaStream_t s = h->stream;
    if (pipelined) {
        // this call runs on the lane's own stream, behind whatever the caller queued so far and behind the lane's
        // previous call (stream order); the handle's stream only joins at dtfill_flush / dtfill_status.
        CU(cudaEventRecord(h->pipe_fork, h->stream));
        s = L->pipe;
        CU(cudaStreamWaitEvent(s, h->pipe_fork, 0));
    } else {
        // strict mode: everything still in flight on the lanes joins the handle's stream first
        for (Lane& o : h->lanes)
            if (o.pending) { CU(cudaStreamWaitEvent(h->stream, o.done, 0)); o.pending = false; }
    }
    int launches = 0;
    // this call's slot of the status ring; a slot that dtfill_status has not examined yet keeps its verdict
    const int slot = h->ncalls % dtfill_ctx::STATUS_RING;
    if (h->slot_dirty[slot]) {
        CU(cudaEventSynchronize(h->slot_done[slot]));
        if (h->status_ring[2 * slot] < h->sticky_bad) h->sticky_bad = h->status_ring[2 * slot];
        if (h->status_ring[2 * slot] != INT_MAX || h->status_ring[2 * slot + 1] != 0) h->slot_rearm[slot] = true;
        h->slot_dirty[slot] = false;
    }
    h->cur_slot = slot;
    h->cur_status = h->status_dev + (size_t)slot * dtfill_ctx::STATUS_STRIDE;
    if (h->slot_rearm[slot] || (h->debug_skip & 2)) {      // (a run without k1b_scan_compact reports nothing)
        CU(cudaMemcpyAsync(h->cur_status, h->status_init, 8, cudaMemcpyHostToDevice, s));
        h->slot_rearm[slot] = false;
    }
    h->cur_status_copied = false;

    // sub-batches on forked streams (skipped while per-kernel profiling is on: the event pairs need one stream)
    int nsub = h->nsub;
    // device-resident data: sub-batches do not pay (the scan is bound by per-task latency).  Host buffers: slices
    // pipeline the PCIe copies in both directions with the kernels.
    if (nsub <= 0) nsub = hio ? (B >= 64 ? 16 : (B >= 32 ? 8 : (B >= 4 ? 4 : 1))) : 1;
    if (nsub > Lane::MAX_SUB) nsub = Lane::MAX_SUB;
    if (nsub > B) nsub = B;
    if (h->profiling || nsub < 1) nsub = 1;
    h->cur_status_early = nsub == 1 && !(h->debug_skip & 2);     // slices share the words: their copy follows the last slice
    void* dense_pin = hio ? hio->in_pin : nullptr;      // pinned mirror of a pageable input (allocated late on the sparse path)
    auto copy_in = [&](cudaStream_t st, int b0, int nb) -> int {
        if (!hio || !hio->in) return 0;
        const size_t frame_bytes = h->in_u16 ? (size_t)h->in_H * W * 2 : (size_t)H * W * 4;
        const char* src = (const char*)hio->in + b0 * frame_bytes;
        if (hio->sparse_pin) {     // pageable float32 input: compact the slice on the host, rebuild it on the device
            const size_t o = (size_t)b0 * H * W, n = (size_t)nb * H * W;
            const size_t cap = n / hio->sparse_cap_div;
            const size_t ro = 2 * (o / hio->sparse_cap_div);          // this slice's region: indices [cap], values [cap]
            uint32_t* pi = hio->sparse_pin + ro;
            uint32_t* pv = pi + cap;
            const size_t cnt = n < (1ull << 32) ? h->pool_in->compact(pi, pv, cap, (const float*)src, n, hio->sparse_scut, hio->sparse_vthr)
                                                : SIZE_MAX;
            if (cnt != SIZE_MAX) {
                float* dst = (float*)const_cast<void*>(in) + o;
                CU(cudaMemsetAsync(dst, 0, n * 4, st));
                if (cnt) {
                    uint32_t* di = (uint32_t*)h->sparse_dev.p + ro;
                    uint32_t* dv = di + cap;
                    CU(cudaMemcpyAsync(di, pi, cnt * 4, cudaMemcpyHostToDevice, st));
                    CU(cudaMemcpyAsync(dv, pv, cnt * 4, cudaMemcpyHostToDevice, st));
                    k0_scatter_pairs<<<(unsigned)((cnt + 255) / 256), 256, 0, st>>>(di, dv, (unsigned)cnt, dst);
                }
                h->last_h2d_bytes += cnt * 8;
                return 0;
            }
            // a slice denser than the pair buffer allows: the mirror after all
            if (!dense_pin) {
                int r = ensure_pinned(h->pin_in, (size_t)B * frame_bytes);
                if (r) return r;
                dense_pin = h->pin_in.p;
            }
        }
        if (dense_pin) {           // pageable input: this slice -> pinned mirror (pool threads), DMA from there
            char* pin = (char*)dense_pin + b0 * frame_bytes;
            h->pool_in->copy(pin, src, nb * frame_bytes);
            src = pin;
        }
        CU(cudaMemcpyAsync((char*)const_cast<void*>(in) + b0 * frame_bytes, src, nb * frame_bytes, cudaMemcpyHostToDevice, st));
        h->last_h2d_bytes += nb * frame_bytes;
        return 0;
    };
    auto copy_out = [&](cudaStream_t st, int b0, int nb) -> int {
        if (!hio) return 0;
        const size_t o = (size_t)b0 * H * W, n = (size_t)nb * H * W;
        CU(cudaMemcpyAsync((hio->depth_pin ? hio->depth_pin : hio->depth) + o, out_depth + o, n * 4, cudaMemcpyDeviceToHost, st));
        if (hio->lidar) CU(cudaMemcpyAsync((hio->lidar_pin ? hio->lidar_pin : hio->lidar) + o, h->lidar_dev + o, n * 4, cudaMemcpyDeviceToHost, st));
        if (hio->dt) CU(cudaMemcpyAsync((hio->dt_pin ? hio->dt_pin : hio->dt) + o, out_dt + o, n * 4, cudaMemcpyDeviceToHost, st));
        if (hio->lbl) CU(cudaMemcpyAsync((hio->lbl_pin ? hio->lbl_pin : hio->lbl) + o, out_lbl + o, n * 4, cudaMemcpyDeviceToHost, st));
        if (hio->mask) CU(cudaMemcpyAsync((hio->mask_pin ? hio->mask_pin : hio->mask) + o, out_mask + o, n, cudaMemcpyDeviceToHost, st));
        if (hio->counts)
            CU(cudaMemcpyAsync(hio->counts + 2 * (size_t)b0, out_counts + 2 * (size_t)b0, (size_t)nb * 8,
                               cudaMemcpyDeviceToHost, st));
        h->last_d2h_bytes += n * (4 + (hio->lidar ? 4 : 0) + (hio->dt ? 4 : 0) + (hio->lbl ? 4 : 0) + (hio->mask ? 1 : 0));
        return 0;
    };
    if (nsub == 1 && !(hio && hio->any_out_pin())) {
        if ((rc = copy_in(s, 0, B))) return rc;
        if ((rc = enqueue_range(h, L, s, plan, 0, B, B, in, H, W, src_thr, val_thr, out_depth, out_dt, out_lbl, out_mask,
                                out_counts, scratch_units_per_frame, 0, &launches))) return rc;
        if ((rc = copy_out(s, 0, B))) return rc;
    } else {
        // pageable outputs: a drain thread waits for each slice's device-to-host copies and moves the slice from the
        // pinned mirrors into the caller's arrays while the later slices are still being copied in and computed
        std::atomic<int> enqueued{0};
        std::atomic<bool> abort_drain{false};
        std::thread drain;
        const bool draining = hio && hio->any_out_pin();
        if (draining) {
            drain = std::thread([&, L] {
                cudaSetDevice(h->device);
                for (int i = 0; i < nsub; ++i) {
                    while (enqueued.load(std::memory_order_acquire) <= i) {
                        if (abort_drain.load()) return;
                        std::this_thread::yield();
                    }
                    if (cudaEventSynchronize(L->join_ev[i]) != cudaSuccess) return;
                    const int b0 = (int)((long)B * i / nsub), b1 = (int)((long)B * (i + 1) / nsub);
                    const size_t o = (size_t)b0 * H * W, n = (size_t)(b1 - b0) * H * W;
                    if (hio->depth_pin) h->pool_out->copy(hio->depth + o, hio->depth_pin + o, n * 4);
                    if (hio->lidar_pin) h->pool_out->copy(hio->lidar + o, hio->lidar_pin + o, n * 4);
                    if (hio->dt_pin) h->pool_out->copy(hio->dt + o, hio->dt_pin + o, n * 4);
                    if (hio->lbl_pin) h->pool_out->copy(hio->lbl + o, hio->lbl_pin + o, n * 4);
                    if (hio->mask_pin) h->pool_out->copy(hio->mask + o, hio->mask_pin + o, n);
                }
            });
        }
        auto body = [&]() -> int {
            CU(cudaEventRecord(L->fork_ev, s));
            for (int i = 0; i < nsub; ++i) {
                const int b0 = (int)((long)B * i / nsub), b1 = (int)((long)B * (i + 1) / nsub);
                CU(cudaStreamWaitEvent(L->sub[i], L->fork_ev, 0));
                int r;
                if ((r = copy_in(L->sub[i], b0, b1 - b0))) return r;
                if ((r = enqueue_range(h, L, L->sub[i], plan, b0, b1 - b0, B, in, H, W, src_thr, val_thr, out_depth, out_dt,
                                       out_lbl, out_mask, out_counts, scratch_units_per_frame, i, &launches))) return r;
                if ((r = copy_out(L->sub[i], b0, b1 - b0))) return r;
                CU(cudaEventRecord(L->join_ev[i], L->sub[i]));
                CU(cudaStreamWaitEvent(s, L->join_ev[i], 0));
                enqueued.store(i + 1, std::memory_order_release);
            }
            return 0;
        };
        rc = body();
        if (rc) abort_drain.store(true);
        if (drain.joinable()) drain.join();
        if (rc) return rc;
    }
    if (h->ev_gt) {
        // evaluation.py:82-123 / :196-239 on the filled depth of this call, on the call's own stream: per-frame metrics,
        // their column sums added to the lane's running totals (eval.py:212-232 `+=`), no host synchronisation
        const long fnpx = (long)H * W;
        int chunks = (int)((fnpx + 16383) / 16384);
        if (chunks < 1) chunks = 1;
        if (chunks > 64) chunks = 64;
        while (chunks > 1 && (((fnpx + chunks - 1) / chunks) & 3)) --chunks;
        if ((rc = ensure(h, L->ev_partial, (size_t)B * chunks * ACC * 8))) return rc;
        if ((rc = ensure(h, L->ev_per_frame, (size_t)B * 9 * 8))) return rc;
        if (!L->ev_totals.p) {
            if ((rc = ensure(h, L->ev_totals, 10 * 8))) return rc;
            CU(cudaMemsetAsync(L->ev_totals.p, 0, 10 * 8, s));
        }
        dim3 grid(chunks, B);
        double* part = (double*)L->ev_partial.p;
        if (h->ev_gt_f64) {
            if (h->ev_mode == 0) k4_metrics_partial<double, 0><<<grid, 256, 0, s>>>(out_depth, (const double*)h->ev_gt, fnpx, chunks, part);
            else k4_metrics_partial<double, 1><<<grid, 256, 0, s>>>(out_depth, (const double*)h->ev_gt, fnpx, chunks, part);
        } else {
            if (h->ev_mode == 0) k4_metrics_partial<float, 0><<<grid, 256, 0, s>>>(out_depth, (const float*)h->ev_gt, fnpx, chunks, part);
            else k4_metrics_partial<float, 1><<<grid, 256, 0, s>>>(out_depth, (const float*)h->ev_gt, fnpx, chunks, part);
        }
        k4_metrics_final<<<1, 256, 0, s>>>(part, B, chunks, h->ev_mode, (double*)L->ev_per_frame.p, (double*)L->ev_totals.p, 1);
        launches += 2;
        L->ev_dirty = true;
    }
    if (!h->cur_status_copied) {
        CU(cudaMemcpyAsync(h->status_ring + 2 * slot, h->cur_status, 8, cudaMemcpyDeviceToHost, s));
        CU(cudaEventRecord(h->slot_done[slot], s));
    }
    h->cur_status_early = false;
    h->slot_dirty[slot] = true;
    h->last_slot = slot;
    CU(cudaGetLastError());
    if (pipelined) {
        CU(cudaEventRecord(L->done, s));
        L->pending = true;
    }
    L->last_launches = launches;
    L->last_B = B;
    h->last_lane = (int)(L - h->lanes);
    ++h->ncalls;
    return 0;
}

// Per-frame metrics in numpy's own summation order (k4x_*): per-pixel terms of the valid pixels compacted in raster order,
// then the pairwise tree of np.add.reduce; groups of frames share a scratch of at most ~4 GiB (a batch of 256 KITTI frames
// with a float64 ground truth needs 3.5 GB: one group, every frame's tree in flight at once).  GT: the arithmetic type,
// GS: the ground truth as stored.  WIN: npx is the area of the crop window `win` of frames of win.frame_px pixels.  Device
// pointers; enqueued on s.
template <typename GT, int MODE, typename GS, bool WIN = false>
int k4x_enqueue(dtfill_t* h, const float* pred, const GS* gt, int B, long npx, double* per_frame, cudaStream_t s,
                const K4xWindow& win = K4xWindow{}) {
    const long fstride = WIN ? win.frame_px : npx;
    const size_t gsz = sizeof(GT);
    const long maxl = npx / 64 + 2;
    long G = (long)((1ull << 32) / ((size_t)4 * npx * gsz));
    G = G < 1 ? 1 : (G > B ? B : G);
    int rc;
    if ((rc = ensure(h, h->mx_terms, (size_t)G * 4 * npx * gsz))) return rc;
    if ((rc = ensure(h, h->mx_counts, (size_t)G * 4 * 4))) return rc;
    if ((rc = ensure(h, h->mx_leaf_start, (size_t)G * maxl * 4))) return rc;
    if ((rc = ensure(h, h->mx_leaf_sum, (size_t)G * 4 * maxl * gsz))) return rc;
    for (long g0 = 0; g0 < B; g0 += G) {
        const int ng = (int)(B - g0 < G ? B - g0 : G);
        GT* tm = (GT*)h->mx_terms.p;
        int* cn = (int*)h->mx_counts.p;
        k4x_compact<GT, MODE, GS, WIN><<<ng, K4X_THREADS, 0, s>>>(pred + g0 * fstride, gt + g0 * fstride, npx, tm, cn, win);
        k4x_reduce<GT><<<ng, K4X_RTHREADS, 0, s>>>(tm, cn, npx, MODE, (int*)h->mx_leaf_start.p, (GT*)h->mx_leaf_sum.p,
                                                   per_frame + g0 * 9);
    }
    return 0;
}

}  // namespace

extern "C" {

int dtfill_abi_version(void) { return DTFILL_ABI_VERSION; }

const char* dtfill_last_error(void) { return g_err.c_str(); }

int dtfill_create(int device, dtfill_t** out_handle) {
    if (!out_handle) return fail(DTFILL_E_ARG, "dtfill_create: NULL out_handle");
    *out_handle = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0)
        return fail(DTFILL_E_CUDA, std::string("dtfill_create: no usable CUDA device (") +
                                       (e != cudaSuccess ? cudaGetErrorString(e) : "count = 0") +
                                       "); this library has no CPU fallback");
    if (device < 0 || device >= n) return fail(DTFILL_E_ARG, "dtfill_create: device index out of range");
    CU(cudaSetDevice(device));
    dtfill_t* h = new (std::nothrow) dtfill_ctx();
    if (!h) return fail(DTFILL_E_NOMEM, "dtfill_create: out of host memory");
    h->device = device;
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    h->sm_count = prop.multiProcessorCount;
    CU(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    h->stream = h->own_stream;
    for (auto& e : h->ev) CU(cudaEventCreate(&e));
    CU(cudaEventCreateWithFlags(&h->pipe_fork, cudaEventDisableTiming));
    CU(cudaHostAlloc((void**)&h->status_ring, dtfill_ctx::STATUS_RING * 8 + 8, cudaHostAllocDefault));
    h->status_init = h->status_ring + 2 * dtfill_ctx::STATUS_RING;
    h->status_init[0] = INT_MAX;
    h->status_init[1] = 0;
    for (auto& e : h->slot_done) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    {
        const size_t n = (size_t)dtfill_ctx::STATUS_RING * dtfill_ctx::STATUS_STRIDE;
        std::vector<int> init(n, 0);
        for (int i = 0; i < dtfill_ctx::STATUS_RING; ++i) init[(size_t)i * dtfill_ctx::STATUS_STRIDE] = INT_MAX;
        CU(cudaMalloc((void**)&h->status_dev, n * sizeof(int)));
        CU(cudaMemcpy(h->status_dev, init.data(), n * sizeof(int), cudaMemcpyHostToDevice));
        CU(cudaStreamCreateWithFlags(&h->status_stream, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&h->status_fork, cudaEventDisableTiming));
    }
    int prio_hi = 0;
    CU(cudaDeviceGetStreamPriorityRange(nullptr, &prio_hi));      // numerically lower = higher priority
    for (Lane& L : h->lanes) {
        CU(cudaStreamCreateWithPriority(&L.pipe, cudaStreamNonBlocking, prio_hi));
        CU(cudaEventCreateWithFlags(&L.done, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&L.fork_ev, cudaEventDisableTiming));
        for (int i = 0; i < Lane::MAX_SUB; ++i) {
            CU(cudaStreamCreateWithFlags(&L.sub[i], cudaStreamNonBlocking));
            CU(cudaEventCreateWithFlags(&L.join_ev[i], cudaEventDisableTiming));
            CU(cudaStreamCreateWithPriority(&L.side[i], cudaStreamNonBlocking, prio_hi));
            CU(cudaEventCreateWithFlags(&L.side_fork[i], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&L.side_join[i], cudaEventDisableTiming));
        }
    }
    if (const char* e = getenv("DTFILL_SUBBATCHES")) h->nsub = atoi(e);
    if (const char* e = getenv("DTFILL_SKY_MIN")) h->sky_min = atoi(e) < -1 ? -1 : atoi(e);
    if (const char* e = getenv("DTFILL_BAND_CAP")) h->band_cap = atoi(e);
    if (const char* e = getenv("DTFILL_STAGE_THREADS")) h->stage_threads = atoi(e);
    if (const char* e = getenv("DTFILL_SPARSE_UPLOAD")) h->sparse_upload = atoi(e) != 0;
    if (const char* e = getenv("DTFILL_METRICS_EXACT")) h->metrics_exact = atoi(e) != 0;
    if (const char* e = getenv("DTFILL_PIPELINE_DEPTH")) {
        const int d = atoi(e);
        h->pipeline_depth = d < 1 ? 1 : (d > dtfill_ctx::MAX_LANES ? dtfill_ctx::MAX_LANES : d);
    }
    *out_handle = h;
    return 0;
}

void dtfill_destroy(dtfill_t* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    for (Lane& L : h->lanes) {
        Buf* lb[] = {&L.srcbits, &L.wprefix, &L.rowcell, &L.rowsrc, &L.rowval, &L.counts, &L.dlist,
                     &L.scratch, &L.tasks, &L.sky, &L.skykeys, &L.ev_partial, &L.ev_per_frame, &L.ev_totals};
        for (Buf* b : lb)
            if (b->p) cudaFree(b->p);
        if (L.fork_ev) cudaEventDestroy(L.fork_ev);
        if (L.done) cudaEventDestroy(L.done);
        if (L.pipe) cudaStreamDestroy(L.pipe);
        for (int i = 0; i < Lane::MAX_SUB; ++i) {
            if (L.join_ev[i]) cudaEventDestroy(L.join_ev[i]);
            if (L.sub[i]) cudaStreamDestroy(L.sub[i]);
            if (L.side_fork[i]) cudaEventDestroy(L.side_fork[i]);
            if (L.side_join[i]) cudaEventDestroy(L.side_join[i]);
            if (L.side[i]) cudaStreamDestroy(L.side[i]);
        }
    }
    Buf* bufs[] = {&h->in_dev, &h->depth_dev, &h->dt_dev, &h->lbl_dev, &h->mask_dev, &h->counts_out_dev, &h->lidar_out_dev,
                   &h->gt_dev, &h->partial, &h->per_frame, &h->sums, &h->edt_rows, &h->edt_stack, &h->sparse_dev,
                   &h->mx_terms, &h->mx_counts, &h->mx_leaf_start, &h->mx_leaf_sum, &h->png_data, &h->png_scratch,
                   &h->png_samples, &h->png_status, &h->enc_in, &h->enc_filt, &h->enc_adler, &h->enc_slots, &h->enc_seg,
                   &h->enc_out, &h->enc_off, &h->enc_depth, &h->smp_coords, &h->smp_bad};
    for (Buf* b : bufs)
        if (b->p) cudaFree(b->p);
    for (void* q : h->retired) cudaFree(q);
    if (h->counts_host) cudaFreeHost(h->counts_host);
    delete h->pool_in;
    delete h->pool_out;
    for (PinBuf* b : {&h->pin_in, &h->pin_depth, &h->pin_dt, &h->pin_lbl, &h->pin_mask, &h->pin_lidar, &h->pin_sparse, &h->pin_png,
                      &h->pin_png_status, &h->pin_enc_off, &h->pin_smp, &h->pin_smp_out})
        if (b->p) cudaFreeHost(b->p);
    if (h->status_ring) cudaFreeHost(h->status_ring);
    if (h->status_dev) cudaFree(h->status_dev);
    if (h->status_stream) cudaStreamDestroy(h->status_stream);
    if (h->status_fork) cudaEventDestroy(h->status_fork);
    for (auto& e : h->slot_done)
        if (e) cudaEventDestroy(e);
    for (auto& e : h->ev)
        if (e) cudaEventDestroy(e);
    if (h->pipe_fork) cudaEventDestroy(h->pipe_fork);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    delete h;
}

// Make the handle's stream wait for every call still in flight on the lanes (pipelined mode).
int dtfill_flush(dtfill_t* h) {
    if (!h) return fail(DTFILL_E_ARG, "dtfill_flush: NULL handle");
    CU(cudaSetDevice(h->device));
    for (Lane& L : h->lanes)
        if (L.pending) { CU(cudaStreamWaitEvent(h->stream, L.done, 0)); L.pending = false; }
    return 0;
}

int dtfill_set_pipeline_depth(dtfill_t* h, int depth) {
    if (!h) return fail(DTFILL_E_ARG, "dtfill_set_pipeline_depth: NULL handle");
    int rc = dtfill_flush(h);
    if (rc) return rc;
    h->pipeline_depth = depth < 1 ? 1 : (depth > dtfill_ctx::MAX_LANES ? dtfill_ctx::MAX_LANES : depth);
    return 0;
}

int dtfill_set_stream(dtfill_t* h, void* cuda_stream) {
    if (!h) return fail(DTFILL_E_ARG, "dtfill_set_stream: NULL handle");
    cudaStream_t ns = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
    if (ns != h->stream) {
        int rc = dtfill_flush(h);          // work in flight joins the stream it was issued against
        if (rc) return rc;
        h->stream = ns;
    }
    return 0;
}

int dtfill_synchronize(dtfill_t* h) {
    if (!h) return fail(DTFILL_E_ARG, "dtfill_synchronize: NULL handle");
    int rc = dtfill_flush(h);
    if (rc) return rc;
    CU(cudaStreamSynchronize(h->stream));
    if (!h->retired.empty()) {            // buffers outgrown by an earlier call: nothing in flight uses them any more
        for (void* q : h->retired) cudaFree(q);
        h->retired.clear();
    }
    return 0;
}

int dtfill_run_async(dtfill_t* h, const float* in_dev, int B, int H, int W, float src_thr, float val_thr,
                     float* out_depth_dev, float* out_dt_dev, int32_t* out_lbl_dev, uint8_t* out_mask_dev,
                     int32_t* out_counts_dev) {
    return enqueue(h, in_dev, B, H, W, src_thr, val_thr, out_depth_dev, out_dt_dev, out_lbl_dev, out_mask_dev,
                   out_counts_dev);
}

int dtfill_status(dtfill_t* h, int* first_bad_frame, int* kernel_launches) {
    if (!h) return fail(DTFILL_E_ARG, "dtfill_status: NULL handle");
    int rc = dtfill_synchronize(h);
    if (rc) return rc;
    CU(cudaStreamSynchronize(h->status_stream));
    if (kernel_launches) *kernel_launches = h->lanes[h->last_lane].last_launches;
    // calls examined: every one since the previous dtfill_status (each has its own slot of the status ring)
    int bad = h->sticky_bad;
    h->sticky_bad = INT_MAX;
    for (int i = 0; i < dtfill_ctx::STATUS_RING; ++i)
        if (h->slot_dirty[i]) {
            if (h->status_ring[2 * i] < bad) bad = h->status_ring[2 * i];
            if (h->status_ring[2 * i] != INT_MAX || h->status_ring[2 * i + 1] != 0) h->slot_rearm[i] = true;
            h->slot_dirty[i] = false;
        }
    if (first_bad_frame) *first_bad_frame = (bad == INT_MAX) ? -1 : bad;
    if (bad != INT_MAX)
        return fail(DTFILL_E_INDEX, "frame " + std::to_string(bad) +
                                        ": labels index outside the list of valid depths (numpy IndexError)");
    return 0;
}

namespace {

// Input description of one call, installed on the handle while the call is enqueued.
struct InputScope {
    dtfill_t* h;
    InputScope(dtfill_t* h_, bool u16, int in_H, int in_crop, float* lidar_dev) : h(h_) {
        h->in_u16 = u16; h->in_H = in_H; h->in_crop = in_crop; h->lidar_dev = lidar_dev;
    }
    ~InputScope() { h->in_u16 = false; h->in_H = 0; h->in_crop = 0; h->lidar_dev = nullptr; }
};

// dtfill_run / dtfill_run_u16: buffers on either side, synchronous.  u16: `in` holds uint16 samples [B,in_H,W].
int run_sync(dtfill_t* h, const void* in, int in_is_device, bool u16, int in_H, int in_crop, int B, int H, int W,
             float src_thr, float val_thr, float* out_lidar, float* out_depth, float* out_dt, int32_t* out_lbl,
             uint8_t* out_mask, int32_t* out_counts, int out_is_device, int* first_bad_frame, bool in_resident = false) {
    CU(cudaSetDevice(h->device));
    const size_t npx = (size_t)B * H * W;
    const size_t in_bytes = u16 ? (size_t)B * in_H * W * 2 : npx * 4;
    int rc;
    const void* in_d = in;
    // outputs on the host: copies are sliced.  in_resident: the input is a device buffer the library itself just produced
    // (dtfill_run_png), so only the outputs go through the slices
    const bool pipelined = !out_is_device && (!in_is_device || in_resident);
    if (!in_is_device) {
        if ((rc = ensure(h, h->in_dev, in_bytes))) return rc;
        if (!pipelined) CU(cudaMemcpyAsync(h->in_dev.p, in, in_bytes, cudaMemcpyHostToDevice, h->stream));
        in_d = h->in_dev.p;
    }
    float* olid = out_lidar; float* od = out_depth; float* odt = out_dt; int32_t* ol = out_lbl; uint8_t* om = out_mask;
    int32_t* oc = out_counts;
    if (!out_is_device) {
        if ((rc = ensure(h, h->depth_dev, npx * 4))) return rc;
        od = (float*)h->depth_dev.p;
        if (out_lidar) { if ((rc = ensure(h, h->lidar_out_dev, npx * 4))) return rc; olid = (float*)h->lidar_out_dev.p; }
        if (out_dt) { if ((rc = ensure(h, h->dt_dev, npx * 4))) return rc; odt = (float*)h->dt_dev.p; }
        if (out_lbl) { if ((rc = ensure(h, h->lbl_dev, npx * 4))) return rc; ol = (int32_t*)h->lbl_dev.p; }
        if (out_mask) { if ((rc = ensure(h, h->mask_dev, npx))) return rc; om = (uint8_t*)h->mask_dev.p; }
        if (out_counts) { if ((rc = ensure(h, h->counts_out_dev, (size_t)B * 8))) return rc; oc = (int32_t*)h->counts_out_dev.p; }
    }
    InputScope scope(h, u16, in_H, in_crop, olid);
    h->last_h2d_bytes = h->last_d2h_bytes = 0;
    if (pipelined) {
        HostIO hio;
        hio.in = in_resident ? nullptr : in; hio.lidar = out_lidar; hio.depth = out_depth; hio.dt = out_dt; hio.lbl = out_lbl; hio.mask = out_mask;
        // pageable buffers go through pinned mirrors (DTFILL_STAGE_THREADS=0 / dtfill_set_stage_threads(h, 0): never)
        if (h->stage_threads != 0) {
            const bool pin_i = !in_resident && is_pageable(in);
            const bool pin_d = is_pageable(out_depth), pin_t = out_dt && is_pageable(out_dt);
            const bool pin_l = out_lbl && is_pageable(out_lbl), pin_m = out_mask && is_pageable(out_mask);
            const bool pin_x = out_lidar && is_pageable(out_lidar);
            if (pin_i || pin_d || pin_t || pin_l || pin_m || pin_x) {
                if (!h->pool_in) {
                    int n = h->stage_threads;
                    if (n < 0) {      // three quarters of the CPUs this process may run on, 2..12 (measured on a 16-CPU
                        cpu_set_t set;    // box: 8 threads 25.5 k frames/s, 12 threads 26.4 k, 16 the same)
                        int avail = (int)std::thread::hardware_concurrency();
                        if (sched_getaffinity(0, sizeof(set), &set) == 0) avail = CPU_COUNT(&set);
                        n = 3 * avail / 4;
                        n = n < 2 ? 2 : (n > 12 ? 12 : n);
                    }
                    h->pool_in = new CopyPool(n - 1);       // the calling thread works too
                    h->pool_out = new CopyPool(n - 1);
                }
                // pageable float32 input whose zero pixels are neither sources nor valid: sparse upload (the dense mirror
                // is only allocated if a slice turns out too dense)
                const float scut = source_cut(src_thr);
                const size_t cap_div = 4;                       // room for 25 % of the pixels
                if (pin_i && !u16 && h->sparse_upload && scut > 0.0f && val_thr >= 0.0f) {
                    if ((rc = ensure_pinned(h->pin_sparse, (npx / cap_div + 16) * 8))) return rc;
                    if ((rc = ensure(h, h->sparse_dev, (npx / cap_div + 16) * 8))) return rc;
                    hio.sparse_pin = (uint32_t*)h->pin_sparse.p;
                    hio.sparse_cap_div = cap_div;
                    hio.sparse_scut = scut; hio.sparse_vthr = val_thr;
                    if (h->pin_in.cap >= in_bytes) hio.in_pin = h->pin_in.p;
                } else if (pin_i) { if ((rc = ensure_pinned(h->pin_in, in_bytes))) return rc; hio.in_pin = h->pin_in.p; }
                if (pin_d) { if ((rc = ensure_pinned(h->pin_depth, npx * 4))) return rc; hio.depth_pin = (float*)h->pin_depth.p; }
                if (pin_t) { if ((rc = ensure_pinned(h->pin_dt, npx * 4))) return rc; hio.dt_pin = (float*)h->pin_dt.p; }
                if (pin_l) { if ((rc = ensure_pinned(h->pin_lbl, npx * 4))) return rc; hio.lbl_pin = (int32_t*)h->pin_lbl.p; }
                if (pin_m) { if ((rc = ensure_pinned(h->pin_mask, npx))) return rc; hio.mask_pin = (uint8_t*)h->pin_mask.p; }
                if (pin_x) { if ((rc = ensure_pinned(h->pin_lidar, npx * 4))) return rc; hio.lidar_pin = (float*)h->pin_lidar.p; }
            }
        }
        if (out_counts) {
            if (h->counts_host_cap < (size_t)B * 2) {
                if (h->counts_host) cudaFreeHost(h->counts_host);
                h->counts_host = nullptr;
                h->counts_host_cap = 0;
                CU(cudaHostAlloc((void**)&h->counts_host, (size_t)B * 8 + 64, cudaHostAllocDefault));
                h->counts_host_cap = (size_t)B * 2 + 16;
            }
            hio.counts = h->counts_host;
        }
        if ((rc = enqueue(h, in_d, B, H, W, src_thr, val_thr, od, odt, ol, om, oc, &hio, true))) return rc;
        rc = dtfill_status(h, first_bad_frame, nullptr);
        if (out_counts && (rc == 0 || rc == DTFILL_E_INDEX)) memcpy(out_counts, h->counts_host, (size_t)B * 8);
        return rc;
    }
    if ((rc = enqueue(h, in_d, B, H, W, src_thr, val_thr, od, odt, ol, om, oc, nullptr, true))) return rc;
    if (!out_is_device) {
        CU(cudaMemcpyAsync(out_depth, od, npx * 4, cudaMemcpyDeviceToHost, h->stream));
        if (out_lidar) CU(cudaMemcpyAsync(out_lidar, olid, npx * 4, cudaMemcpyDeviceToHost, h->stream));
        if (out_dt) CU(cudaMemcpyAsync(out_dt, odt, npx * 4, cudaMemcpyDeviceToHost, h->stream));
        if (out_lbl) CU(cudaMemcpyAsync(out_lbl, ol, npx * 4, cudaMemcpyDeviceToHost, h->stream));
        if (out_mask) CU(cudaMemcpyAsync(out_mask, om, npx, cudaMemcpyDeviceToHost, h->stream));
        if (out_counts) CU(cudaMemcpyAsync(out_counts, oc, (size_t)B * 8, cudaMemcpyDeviceToHost, h->stream));
    }
    return dtfill_status(h, first_bad_frame, nullptr);
}

int check_u16_args(const char* who, dtfill_t* h, const void* in, const void* out_depth, int B, int in_H, int W, int crop_top) {
    if (!h || !in || !out_depth) return fail(DTFILL_E_ARG, std::string(who) + ": NULL handle, input or out_depth");
    if (B <= 0 || in_H <= 0 || W <= 0) return fail(DTFILL_E_ARG, std::string(who) + ": B, H_in, W must be positive");
    if (crop_top < 0 || crop_top >= in_H) return fail(DTFILL_E_ARG, std::string(who) + ": crop_top must lie in [0, H_in)");
    return 0;
}

}  // namespace

int dtfill_run(dtfill_t* h, const float* in, int in_is_device, int B, int H, int W, float src_thr, float val_thr,
               float* out_depth, float* out_dt, int32_t* out_lbl, uint8_t* out_mask, int32_t* out_counts,
               int out_is_device, int* first_bad_frame) {
    if (first_bad_frame) *first_bad_frame = -1;
    if (!h || !in || !out_depth) return fail(DTFILL_E_ARG, "dtfill_run: NULL handle, input or out_depth");
    if (B <= 0 || H <= 0 || W <= 0) return fail(DTFILL_E_ARG, "dtfill_run: B, H, W must be positive");
    return run_sync(h, in, in_is_device, false, H, 0, B, H, W, src_thr, val_thr, nullptr, out_depth, out_dt, out_lbl,
                    out_mask, out_counts, out_is_device, first_bad_frame);
}

int dtfill_run_u16(dtfill_t* h, const uint16_t* in, int in_is_device, int B, int H_in, int W, int crop_top, float src_thr,
                   float val_thr, float* out_lidar, float* out_depth, float* out_dt, int32_t* out_lbl, uint8_t* out_mask,
                   int32_t* out_counts, int out_is_device, int* first_bad_frame) {
    if (first_bad_frame) *first_bad_frame = -1;
    int rc = check_u16_args("dtfill_run_u16", h, in, out_depth, B, H_in, W, crop_top);
    if (rc) return rc;
    return run_sync(h, in, in_is_device, true, H_in, crop_top, B, H_in - crop_top, W, src_thr, val_thr, out_lidar, out_depth,
                    out_dt, out_lbl, out_mask, out_counts, out_is_device, first_bad_frame);
}

int dtfill_run_u16_async(dtfill_t* h, const uint16_t* in_dev, int B, int H_in, int W, int crop_top, float src_thr,
                         float val_thr, float* out_lidar_dev, float* out_depth_dev, float* out_dt_dev, int32_t* out_lbl_dev,
                         uint8_t* out_mask_dev, int32_t* out_counts_dev) {
    int rc = check_u16_args("dtfill_run_u16_async", h, in_dev, out_depth_dev, B, H_in, W, crop_top);
    if (rc) return rc;
    InputScope scope(h, true, H_in, crop_top, out_lidar_dev);
    return enqueue(h, in_dev, B, H_in - crop_top, W, src_thr, val_thr, out_depth_dev, out_dt_dev, out_lbl_dev, out_mask_dev,
                   out_counts_dev);
}

// ------------------------------------------------------------------------------------------------------------
// 16-bit grayscale PNG files -> uint16 samples (k8_png_inflate, k8_png_unfilter; see dtfill_k8_png.cuh)
// ------------------------------------------------------------------------------------------------------------
namespace {

const char* png_reason(int st) {
    switch (st) {
        case png::ST_SIGNATURE: return "bad PNG signature";
        case png::ST_IHDR: return "unsupported IHDR (only non-interlaced 16-bit grayscale PNGs are supported)";
        case png::ST_SIZE: return "image size differs from the batch's";
        case png::ST_CHUNKS: return "broken or truncated chunk structure, or no IDAT";
        case png::ST_ZLIB: return "bad zlib header";
        case png::ST_DEFLATE: return "invalid DEFLATE data";
        case png::ST_LENGTH: return "decompressed size differs from H*(1+2W)";
        case png::ST_FILTER: return "row filter type > 4";
        case png::ST_ADLER: return "Adler-32 mismatch";
        default: return "unknown status";
    }
}

int png_args(const char* who, dtfill_t* h, const void* data, const int64_t* offsets, const void* out, int B, int H, int W) {
    if (!h || !data || !offsets || !out) return fail(DTFILL_E_ARG, std::string(who) + ": NULL handle, data, offsets or output");
    if (B <= 0 || H <= 0 || W <= 0) return fail(DTFILL_E_ARG, std::string(who) + ": B, H, W must be positive");
    // the Adler-32 sums of k8_png_inflate are exact in 64 bits below this size
    if ((int64_t)H * (1 + 2 * (int64_t)W) >= (1ll << 28))
        return fail(DTFILL_E_ARG, std::string(who) + ": frame too large (H * (1 + 2 W) < 2^28 bytes)");
    return 0;
}

// First failed frame of a host copy of the per-frame status: DTFILL_E_DATA with the frame and the reason, or 0.
int png_verdict(const int32_t* st, int B, int* first_bad_frame) {
    for (int b = 0; b < B; ++b)
        if (st[b] != png::ST_OK) {
            if (first_bad_frame) *first_bad_frame = b;
            return fail(DTFILL_E_DATA, "frame " + std::to_string(b) + ": " + png_reason(st[b]) + " (status " +
                                           std::to_string(st[b]) + ")");
        }
    return 0;
}

// One set of host files: file b = data[offsets[b], offsets[b+1]), b < B.
struct PngFiles { const uint8_t* data; const int64_t* offsets; int B; };

// Stage sets of host files into the pinned buffer, back to back in the order given (bytes, then the offsets of all of
// them rebased to 0), and enqueue one copy of it to the device.  The caller waits for the call before the buffer is used
// again.
int png_stage(dtfill_t* h, const PngFiles* sets, int nsets, const uint8_t** d_data, const int64_t** d_off) {
    int rc;
    size_t nbytes = 0;
    int nfiles = 0;
    for (int k = 0; k < nsets; ++k) {
        const PngFiles& f = sets[k];
        if (f.offsets[0] < 0) return fail(DTFILL_E_ARG, "dtfill_png_decode: offsets[0] < 0");
        for (int b = 0; b < f.B; ++b)
            if (f.offsets[b + 1] < f.offsets[b]) return fail(DTFILL_E_ARG, "dtfill_png_decode: offsets decrease at file " + std::to_string(b));
        nbytes += (size_t)(f.offsets[f.B] - f.offsets[0]);
        nfiles += f.B;
    }
    const size_t off_at = (nbytes + 15) & ~(size_t)15;
    const size_t total = off_at + (size_t)(nfiles + 1) * 8;
    if ((rc = ensure_pinned(h->pin_png, total))) return rc;
    if ((rc = ensure(h, h->png_data, total))) return rc;
    uint8_t* pin = (uint8_t*)h->pin_png.p;
    int64_t* po = (int64_t*)(pin + off_at);
    int64_t pos = 0;
    int i = 0;
    for (int k = 0; k < nsets; ++k) {
        const PngFiles& f = sets[k];
        const int64_t o0 = f.offsets[0];
        memcpy(pin + pos, f.data + o0, (size_t)(f.offsets[f.B] - o0));
        for (int b = 0; b < f.B; ++b) po[i++] = pos + f.offsets[b] - o0;
        pos += f.offsets[f.B] - o0;
    }
    po[i] = pos;
    CU(cudaMemcpyAsync(h->png_data.p, pin, total, cudaMemcpyHostToDevice, h->stream));
    h->last_h2d_bytes = total;
    *d_data = (const uint8_t*)h->png_data.p;
    *d_off = (const int64_t*)((uint8_t*)h->png_data.p + off_at);
    return 0;
}

// Enqueue the decode of B files on the handle's stream: samples into out_dev [B,H,W], status into status_dev [B].  Host
// files go up in one copy through the pinned staging buffer (png_stage).
int png_enqueue(dtfill_t* h, const uint8_t* data, const int64_t* offsets, int in_is_device, int B, int H, int W,
                uint16_t* out_dev, int32_t* status_dev) {
    int rc;
    const uint8_t* d_data = data;
    const int64_t* d_off = offsets;
    if (!in_is_device) {
        const PngFiles set{data, offsets, B};
        if ((rc = png_stage(h, &set, 1, &d_data, &d_off))) return rc;
    }
    const size_t fbytes = (size_t)H * (1 + 2 * (size_t)W);
    if ((rc = ensure(h, h->png_scratch, (size_t)B * fbytes))) return rc;
    const int grid = (B + png::K8_WARPS - 1) / png::K8_WARPS;
    uint8_t* scr = (uint8_t*)h->png_scratch.p;
    png::k8_png_inflate<<<grid, 32 * png::K8_WARPS, 0, h->stream>>>(d_data, d_off, B, H, W, scr, status_dev);
    png::k8_png_unfilter<<<grid, 32 * png::K8_WARPS, 0, h->stream>>>(scr, B, H, W, out_dev, status_dev);
    CU(cudaGetLastError());
    return 0;
}

int png_status_host(dtfill_t* h, int B, int32_t** out) {
    int rc = ensure_pinned(h->pin_png_status, (size_t)B * 4);
    if (rc) return rc;
    *out = (int32_t*)h->pin_png_status.p;
    return 0;
}

}  // namespace

int dtfill_png_decode(dtfill_t* h, const uint8_t* data, const int64_t* offsets, int in_is_device, int B, int H, int W,
                      uint16_t* out, int32_t* out_status, int out_is_device, int* first_bad_frame) {
    if (first_bad_frame) *first_bad_frame = -1;
    int rc = png_args("dtfill_png_decode", h, data, offsets, out, B, H, W);
    if (rc) return rc;
    if (out_is_device && !out_status) return fail(DTFILL_E_ARG, "dtfill_png_decode: out_status is required with device outputs");
    CU(cudaSetDevice(h->device));
    uint16_t* od = out;
    int32_t* os = out_status;
    if (!out_is_device) {
        if ((rc = ensure(h, h->png_samples, (size_t)B * H * W * 2))) return rc;
        if ((rc = ensure(h, h->png_status, (size_t)B * 4))) return rc;
        od = (uint16_t*)h->png_samples.p;
        os = (int32_t*)h->png_status.p;
    }
    if ((rc = png_enqueue(h, data, offsets, in_is_device, B, H, W, od, os))) return rc;
    if (in_is_device && out_is_device) return 0;
    int32_t* st_host = nullptr;
    if ((rc = png_status_host(h, B, &st_host))) return rc;
    if (!out_is_device) CU(cudaMemcpyAsync(out, od, (size_t)B * H * W * 2, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(st_host, os, (size_t)B * 4, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    if (!out_is_device && out_status) memcpy(out_status, st_host, (size_t)B * 4);
    return png_verdict(st_host, B, first_bad_frame);
}

int dtfill_run_png(dtfill_t* h, const uint8_t* data, const int64_t* offsets, int in_is_device, int B, int H_in, int W,
                   int crop_top, float src_thr, float val_thr, float* out_lidar, float* out_depth, float* out_dt,
                   int32_t* out_lbl, uint8_t* out_mask, int32_t* out_counts, int out_is_device, int* first_bad_frame) {
    if (first_bad_frame) *first_bad_frame = -1;
    int rc = png_args("dtfill_run_png", h, data, offsets, out_depth, B, H_in, W);
    if (rc) return rc;
    if ((rc = check_u16_args("dtfill_run_png", h, data, out_depth, B, H_in, W, crop_top))) return rc;
    CU(cudaSetDevice(h->device));
    if ((rc = ensure(h, h->png_samples, (size_t)B * H_in * W * 2))) return rc;
    if ((rc = ensure(h, h->png_status, (size_t)B * 4))) return rc;
    int32_t* st_host = nullptr;
    if ((rc = png_status_host(h, B, &st_host))) return rc;
    uint16_t* samples = (uint16_t*)h->png_samples.p;
    if ((rc = png_enqueue(h, data, offsets, in_is_device, B, H_in, W, samples, (int32_t*)h->png_status.p))) return rc;
    CU(cudaMemcpyAsync(st_host, h->png_status.p, (size_t)B * 4, cudaMemcpyDeviceToHost, h->stream));
    const size_t h2d = in_is_device ? 0 : h->last_h2d_bytes;
    // the fill of dtfill_run_u16 on the decoded samples; it ends with a synchronisation, so st_host is final afterwards
    rc = run_sync(h, samples, 1, true, H_in, crop_top, B, H_in - crop_top, W, src_thr, val_thr, out_lidar, out_depth, out_dt,
                  out_lbl, out_mask, out_counts, out_is_device, first_bad_frame, true);
    h->last_h2d_bytes += h2d;
    if (rc != 0 && rc != DTFILL_E_INDEX) return rc;
    const int rd = png_verdict(st_host, B, first_bad_frame);     // a decode failure wins over IndexError
    return rd ? rd : rc;
}

int dtfill_debug_png_decode_host(const uint8_t* f, long nbytes, int H, int W, uint16_t* out) {
    using namespace png;
    if (!f || !out || nbytes < 0 || H <= 0 || W <= 0 || (int64_t)H * (1 + 2 * (int64_t)W) >= (1ll << 28)) return -1;
    const uint32_t total = (uint32_t)H * (uint32_t)(1 + 2 * W);
    std::vector<uint8_t> scr(total);
    std::vector<uint16_t> llut(1 << LBITS), dlut(1 << DBITS);
    uint16_t lsym[288], dsym[32], lcount[16], dcount[16];
    uint32_t qlen[QCAP], qarg[QCAP];
    uint8_t lit[LITCAP], lens[19 + 320];
    Huff lh{llut.data(), lcount, lsym, LBITS}, dh{dlut.data(), dcount, dsym, DBITS};
    Queue q{qlen, qarg, lit, 0, 0};
    Inflate s{};
    int64_t first = 0;
    int st = check_structure(f, nbytes, H, W, &first);
    if (st == ST_OK) {
        idat_open(s.b.in, f, first);
        s.total = total;
        st = zlib_header(s);
    }
    uint32_t p = 0;
    while (st == ST_OK) {
        st = inflate_tokens(s, lh, dh, lens, q);
        for (int i = 0; i < q.n; ++i) {
            const uint32_t len = qlen[i], arg = qarg[i];
            if (arg & LIT_RUN) memcpy(&scr[p], lit + (arg & 0xffff), len);
            else for (uint32_t j = 0; j < len; ++j) scr[p + j] = scr[p - arg + j];
            p += len;
        }
        if (s.state == 3) break;
    }
    if (st == ST_OK) st = finish(s);
    if (st == ST_OK) {
        uint32_t a = 1, bsum = 0;
        for (uint32_t i = 0; i < total; ++i) { a = (a + scr[i]) % ADLER_MOD; bsum = (bsum + a) % ADLER_MOD; }
        if (((bsum << 16) | a) != s.adler) st = ST_ADLER;
    }
    const size_t stride = 1 + 2 * (size_t)W;
    if (st == ST_OK)
        for (int r = 0; r < H; ++r)
            if (scr[r * stride] > 4) { st = ST_FILTER; break; }
    if (st != ST_OK) {
        memset(out, 0, (size_t)H * W * 2);
        return st;
    }
    for (int r = 0; r < H; ++r) {
        const uint8_t* row = &scr[r * stride];
        const int ft = row[0];
        uint16_t* o = out + (size_t)r * W;
        const uint16_t* up = r ? o - W : nullptr;
        for (int c = 0; c < W; ++c) {
            const uint32_t a = c ? o[c - 1] : 0, b = up ? up[c] : 0, cc = (up && c) ? up[c - 1] : 0;
            o[c] = (uint16_t)unfilter_sample(ft, row[1 + 2 * c], row[2 + 2 * c], a, b, cc);
        }
    }
    return ST_OK;
}

// ------------------------------------------------------------------------------------------------------------
// uint16 samples / float32 depth -> 16-bit grayscale PNG files (k9_png_*; see dtfill_k9_png_encode.cuh)
// ------------------------------------------------------------------------------------------------------------
namespace {

int png_encode_args(const char* who, dtfill_t* h, const void* in, const void* out, const int64_t* out_offsets, int B,
                    int H, int W, int64_t out_capacity) {
    if (!h || !in || !out || !out_offsets) return fail(DTFILL_E_ARG, std::string(who) + ": NULL handle, input, out or out_offsets");
    if (B <= 0 || H <= 0 || W <= 0) return fail(DTFILL_E_ARG, std::string(who) + ": B, H, W must be positive");
    if ((int64_t)H * (1 + 2 * (int64_t)W) >= (1ll << 28))
        return fail(DTFILL_E_ARG, std::string(who) + ": frame too large (H * (1 + 2 W) < 2^28 bytes)");
    const int64_t need = (int64_t)B * png::encode_bound(H, W);
    if (out_capacity < need)
        return fail(DTFILL_E_ARG, std::string(who) + ": out_capacity " + std::to_string(out_capacity) + " < B * bound = " +
                                      std::to_string(need));
    return 0;
}

// Enqueue the encode of B device frames (uint16, or float32 depth when is_float) on the handle's stream: the files
// back to back into out_dev, their offsets into off_dev [B+1].
int png_encode_enqueue(dtfill_t* h, const void* in_dev, bool is_float, int B, int H, int W, uint8_t* out_dev,
                       int64_t* off_dev) {
    using namespace png;
    int rc;
    const int64_t stride = 1 + 2 * (int64_t)W, fbytes = (int64_t)H * stride;
    const int nseg = segments(H);
    // a slot holds the chunk header, the larger of the stored form and what the coded form writes before it gives up
    // (at most one batch of tokens, 124 bytes, past the stored size), and the CRC
    const int64_t slot = (8 + stored_bytes((int64_t)(H < SEG_ROWS ? H : SEG_ROWS) * stride) + 256 + 15) & ~(int64_t)15;
    if ((rc = ensure(h, h->enc_filt, (size_t)B * fbytes))) return rc;
    if ((rc = ensure(h, h->enc_adler, (size_t)B * H * 4))) return rc;
    if ((rc = ensure(h, h->enc_slots, (size_t)B * nseg * slot))) return rc;
    if ((rc = ensure(h, h->enc_seg, (size_t)B * nseg * 4))) return rc;
    uint8_t* filt = (uint8_t*)h->enc_filt.p;
    uint32_t* adler = (uint32_t*)h->enc_adler.p;
    uint8_t* slots = (uint8_t*)h->enc_slots.p;
    uint32_t* seg = (uint32_t*)h->enc_seg.p;
    const int64_t rows = (int64_t)B * H;
    const unsigned fgrid = (unsigned)((rows + K9_WARPS - 1) / K9_WARPS);
    if (is_float)
        k9_png_filter<float><<<fgrid, 32 * K9_WARPS, 0, h->stream>>>((const float*)in_dev, B, H, W, filt, adler);
    else
        k9_png_filter<uint16_t><<<fgrid, 32 * K9_WARPS, 0, h->stream>>>((const uint16_t*)in_dev, B, H, W, filt, adler);
    const size_t smem = 256 * 4 + K9_WARPS * sizeof(DeflateSmem);
    CU(cudaFuncSetAttribute(k9_png_deflate, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const unsigned dgrid = (unsigned)(((int64_t)B * nseg + K9_WARPS - 1) / K9_WARPS);
    k9_png_deflate<<<dgrid, 32 * K9_WARPS, smem, h->stream>>>(filt, B, H, W, slots, slot, seg);
    k9_png_offsets<<<1, 1024, 0, h->stream>>>(seg, B, nseg, off_dev);
    k9_png_pack<<<(unsigned)((int64_t)B * (nseg + 2)), 256, 0, h->stream>>>(slots, slot, seg, adler, B, H, W, off_dev, out_dev);
    CU(cudaGetLastError());
    return 0;
}

// dtfill_png_encode / dtfill_png_encode_depth
int png_encode_call(const char* who, dtfill_t* h, const void* in, bool is_float, int in_is_device, int B, int H, int W,
                    uint8_t* out, int64_t out_capacity, int64_t* out_offsets, int out_is_device) {
    int rc = png_encode_args(who, h, in, out, out_offsets, B, H, W, out_capacity);
    if (rc) return rc;
    CU(cudaSetDevice(h->device));
    h->last_h2d_bytes = h->last_d2h_bytes = 0;
    const void* in_d = in;
    if (!in_is_device) {
        const size_t in_bytes = (size_t)B * H * W * (is_float ? 4 : 2);
        if ((rc = ensure(h, h->enc_in, in_bytes))) return rc;
        CU(cudaMemcpyAsync(h->enc_in.p, in, in_bytes, cudaMemcpyHostToDevice, h->stream));
        h->last_h2d_bytes = in_bytes;
        in_d = h->enc_in.p;
    }
    uint8_t* out_d = out;
    int64_t* off_d = out_offsets;
    if (!out_is_device) {
        if ((rc = ensure(h, h->enc_out, (size_t)B * png::encode_bound(H, W)))) return rc;
        if ((rc = ensure(h, h->enc_off, (size_t)(B + 1) * 8))) return rc;
        out_d = (uint8_t*)h->enc_out.p;
        off_d = (int64_t*)h->enc_off.p;
    }
    if ((rc = png_encode_enqueue(h, in_d, is_float, B, H, W, out_d, off_d))) return rc;
    if (in_is_device && out_is_device) return 0;
    if (out_is_device) {
        CU(cudaStreamSynchronize(h->stream));
        return 0;
    }
    // offsets first, then exactly offsets[B] bytes of files
    if ((rc = ensure_pinned(h->pin_enc_off, (size_t)(B + 1) * 8))) return rc;
    int64_t* off_h = (int64_t*)h->pin_enc_off.p;
    CU(cudaMemcpyAsync(off_h, off_d, (size_t)(B + 1) * 8, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    memcpy(out_offsets, off_h, (size_t)(B + 1) * 8);
    CU(cudaMemcpyAsync(out, out_d, (size_t)off_h[B], cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    h->last_d2h_bytes = (size_t)(B + 1) * 8 + (size_t)off_h[B];
    return 0;
}

// The deflate of segment f[s0, s1) run serially: the candidates, parse, codes and fallback of k9_png_deflate.  Writes
// the segment's compressed bytes to out (capacity >= 2 (s1 - s0) + 64) and returns their number.
int64_t png_deflate_segment_host(const uint8_t* f, int64_t s0, int64_t s1, int64_t stride, bool final_seg, uint8_t* out,
                                 uint32_t* head) {
    using namespace png;
    for (int i = 0; i < HSIZE; ++i) head[i] = NO_POS;
    memset(out, 0, (size_t)(2 * (s1 - s0) + 64));
    uint64_t bitpos = 0;
    auto put = [&](uint32_t v, int n) {
        for (int i = 0; i < n; ++i, ++bitpos)
            if ((v >> i) & 1) out[bitpos >> 3] |= (uint8_t)(1u << (bitpos & 7));
    };
    put(2, 3);                                      // BFINAL 0, BTYPE 01
    const int64_t hash_end = s1 - 2;
    int64_t hashed = s0;
    for (int64_t p = s0; p < s1;) {
        for (; hashed < p; ++hashed)
            if (hashed < hash_end) head[hash3(f + hashed)] = (uint32_t)hashed;
        const uint32_t qh = p < hash_end ? head[hash3(f + p)] : NO_POS;
        const int maxlen = (int)((s1 - p) < MAX_MATCH ? s1 - p : MAX_MATCH);
        int best_len = 0;
        int64_t best_d = 0;
        if (maxlen >= 3) {
            const int64_t dist[4] = {1, 2, stride, qh != NO_POS ? p - (int64_t)qh : 0};
            for (int c = 0; c < 4; ++c) {
                if (!(dist[c] > 0 && dist[c] <= p && dist[c] <= WINDOW)) continue;
                const int n = match_len(f, p, dist[c], maxlen);
                if (n >= 3 && (n > best_len || (n == best_len && dist[c] < best_d))) { best_len = n; best_d = dist[c]; }
            }
        }
        uint32_t bits;
        const int nb = token_bits((uint32_t)best_len, best_len ? (uint32_t)best_d : f[p], &bits);
        put(bits, nb);
        p += best_len ? best_len : 1;
    }
    put(0, 7);                                      // end of block
    put(final_seg ? 1 : 0, 3);                      // empty stored block
    bitpos = (bitpos + 7) & ~(uint64_t)7;
    put(0xffff0000u, 32);
    const int64_t nbytes = (int64_t)(bitpos >> 3);
    if (nbytes <= stored_bytes(s1 - s0)) return nbytes;
    return write_stored(f, s0, s1, final_seg, out, 0, 1);
}

}  // namespace

int64_t dtfill_png_encode_bound(int H, int W) {
    if (H <= 0 || W <= 0 || (int64_t)H * (1 + 2 * (int64_t)W) >= (1ll << 28)) return DTFILL_E_ARG;
    return png::encode_bound(H, W);
}

int dtfill_png_encode(dtfill_t* h, const uint16_t* in, int in_is_device, int B, int H, int W, uint8_t* out,
                      int64_t out_capacity, int64_t* out_offsets, int out_is_device) {
    return png_encode_call("dtfill_png_encode", h, in, false, in_is_device, B, H, W, out, out_capacity, out_offsets,
                           out_is_device);
}

int dtfill_png_encode_depth(dtfill_t* h, const float* in, int in_is_device, int B, int H, int W, uint8_t* out,
                            int64_t out_capacity, int64_t* out_offsets, int out_is_device) {
    return png_encode_call("dtfill_png_encode_depth", h, in, true, in_is_device, B, H, W, out, out_capacity, out_offsets,
                           out_is_device);
}

int dtfill_run_png_to_png(dtfill_t* h, const uint8_t* data, const int64_t* offsets, int in_is_device, int B, int H_in,
                          int W, int crop_top, float src_thr, float val_thr, uint8_t* out, int64_t out_capacity,
                          int64_t* out_offsets, int out_is_device, int* first_bad_frame) {
    if (first_bad_frame) *first_bad_frame = -1;
    if (!h || !data || !offsets) return fail(DTFILL_E_ARG, "dtfill_run_png_to_png: NULL handle, data or offsets");
    if (B <= 0 || H_in <= 0 || W <= 0) return fail(DTFILL_E_ARG, "dtfill_run_png_to_png: B, H_in, W must be positive");
    if (crop_top < 0 || crop_top >= H_in) return fail(DTFILL_E_ARG, "dtfill_run_png_to_png: crop_top must lie in [0, H_in)");
    const int H = H_in - crop_top;
    int rc = png_encode_args("dtfill_run_png_to_png", h, data, out, out_offsets, B, H, W, out_capacity);
    if (rc) return rc;
    CU(cudaSetDevice(h->device));
    if ((rc = ensure(h, h->enc_depth, (size_t)B * H * W * 4))) return rc;
    float* depth = (float*)h->enc_depth.p;
    const int run = dtfill_run_png(h, data, offsets, in_is_device, B, H_in, W, crop_top, src_thr, val_thr, nullptr, depth,
                                   nullptr, nullptr, nullptr, nullptr, 1, first_bad_frame);
    if (run != 0 && run != DTFILL_E_INDEX && run != DTFILL_E_DATA) return run;
    const std::string verdict = g_err;
    const size_t h2d = h->last_h2d_bytes;
    if ((rc = png_encode_call("dtfill_run_png_to_png", h, depth, true, 1, B, H, W, out, out_capacity, out_offsets,
                              out_is_device)))
        return rc;
    if (out_is_device) CU(cudaStreamSynchronize(h->stream));
    h->last_h2d_bytes = h2d;
    if (run) g_err = verdict;
    return run;
}

int dtfill_debug_depth_samples_host(const float* depth, long n, uint16_t* out) {
    if (!depth || !out || n < 0) return -1;
    for (long i = 0; i < n; ++i) out[i] = (uint16_t)png::depth_sample(depth[i]);
    return 0;
}

long dtfill_debug_png_encode_host(const uint16_t* samples, int H, int W, uint8_t* out, long capacity) {
    using namespace png;
    if (!samples || !out || H <= 0 || W <= 0 || (int64_t)H * (1 + 2 * (int64_t)W) >= (1ll << 28)) return -1;
    if (capacity < encode_bound(H, W)) return -1;
    const int64_t stride = 1 + 2 * (int64_t)W;
    std::vector<uint8_t> filt((size_t)H * stride);
    for (int r = 0; r < H; ++r) {
        const uint16_t* x = samples + (size_t)r * W;
        const uint16_t* up = r ? x - W : nullptr;
        auto sample = [&](int ft, int c) {
            return filter_sample(ft, x[c], c ? x[c - 1] : 0, up ? up[c] : 0, (up && c) ? up[c - 1] : 0);
        };
        int best = 0;
        unsigned long long best_cost = 0;
        for (int ft = 0; ft < 5; ++ft) {
            unsigned long long cost = 0;
            for (int c = 0; c < W; ++c) {
                const uint32_t y = sample(ft, c);
                cost += msad(y >> 8) + msad(y & 255);
            }
            if (ft == 0 || cost < best_cost) { best = ft; best_cost = cost; }
        }
        uint8_t* o = &filt[(size_t)r * stride];
        o[0] = (uint8_t)best;
        for (int c = 0; c < W; ++c) {
            const uint32_t y = sample(best, c);
            o[1 + 2 * c] = (uint8_t)(y >> 8);
            o[2 + 2 * c] = (uint8_t)y;
        }
    }
    uint32_t tab[256];
    for (uint32_t i = 0; i < 256; ++i) tab[i] = crc_table_entry(i);
    uint32_t a = 1, bsum = 0;
    for (uint8_t v : filt) { a = (a + v) % ADLER_MOD; bsum = (bsum + a) % ADLER_MOD; }
    std::vector<uint32_t> head(HSIZE);
    std::vector<uint8_t> seg;
    write_head(out, tab, H, W);
    int64_t pos = HEAD_BYTES;
    const int nseg = segments(H);
    for (int s = 0; s < nseg; ++s) {
        int64_t s0, s1;
        segment_range(s, H, stride, &s0, &s1);
        seg.resize((size_t)(2 * (s1 - s0) + 64));
        const int64_t n = png_deflate_segment_host(filt.data(), s0, s1, stride, s == nseg - 1, seg.data(), head.data());
        put_be32(out + pos, (uint32_t)n);
        put_be32(out + pos + 4, T_IDAT);
        memcpy(out + pos + 8, seg.data(), (size_t)n);
        put_be32(out + pos + 8 + n, crc32_bytes(tab, 0, out + pos + 4, n + 4));
        pos += 12 + n;
    }
    write_tail(out + pos, tab, (bsum << 16) | a);
    return (long)(pos + TAIL_BYTES);
}

namespace {
struct LaneTotals { const double* p[dtfill_ctx::MAX_LANES]; };
__global__ void k4_fold_totals(LaneTotals lanes, double* __restrict__ sums, int accumulate) {
    const int i = threadIdx.x;
    if (i >= 10) return;
    double s = accumulate ? sums[i] : 0.0;
    for (int l = 0; l < dtfill_ctx::MAX_LANES; ++l)
        if (lanes.p[l]) s += lanes.p[l][i];       // fixed order: lane 0, 1, 2, 3
    sums[i] = s;
}
struct EvalScope {
    dtfill_t* h;
    EvalScope(dtfill_t* h_, const void* gt, int f64, int mode) : h(h_) { h->ev_gt = gt; h->ev_gt_f64 = f64; h->ev_mode = mode; }
    ~EvalScope() { h->ev_gt = nullptr; }
};

// Distance_Transform's verdict on the frames of a synchronous fill, frame by frame as the evaluation loop meets them: rc and
// fill_bad are what dtfill_status reported, cnt the fill's counts [B][2].  `what` names a frame in the message.
int fill_verdict(int rc, int fill_bad, const int32_t* cnt, int B, const char* what, int* first_bad_frame) {
    const int lim = rc == DTFILL_E_INDEX ? fill_bad : B;
    for (int b = 0; b < lim; ++b)
        if (cnt[2 * b + 1] == 1) {
            // eval_NYU.py:126 np.squeeze(lidar[with_value]) makes a single valid depth 0-dimensional; :128 then fails
            if (first_bad_frame) *first_bad_frame = b;
            return fail(DTFILL_E_INDEX, what + std::to_string(b) +
                                            ": one valid depth (numpy IndexError: too many indices for array: array is "
                                            "0-dimensional, but 1 were indexed)");
        }
    if (rc == DTFILL_E_INDEX) {
        if (first_bad_frame) *first_bad_frame = fill_bad;
        return fail(DTFILL_E_INDEX, what + std::to_string(fill_bad) +
                                        ": labels index outside the list of valid depths (numpy IndexError)");
    }
    return 0;
}
}  // namespace

int dtfill_run_eval_async(dtfill_t* h, const float* in_dev, const void* gt_dev, int gt_is_f64, int B, int H, int W,
                          float src_thr, float val_thr, int mode, float* out_depth_dev, float* out_dt_dev,
                          int32_t* out_lbl_dev, uint8_t* out_mask_dev, int32_t* out_counts_dev) {
    if (!h || !gt_dev) return fail(DTFILL_E_ARG, "dtfill_run_eval_async: NULL handle or ground truth");
    if (mode != DTFILL_METRICS_KITTI && mode != DTFILL_METRICS_NYU) return fail(DTFILL_E_ARG, "dtfill_run_eval_async: bad mode");
    EvalScope scope(h, gt_dev, gt_is_f64, mode);
    return enqueue(h, in_dev, B, H, W, src_thr, val_thr, out_depth_dev, out_dt_dev, out_lbl_dev, out_mask_dev,
                   out_counts_dev);
}

int dtfill_eval_totals(dtfill_t* h, double* sums_dev, int accumulate) {
    if (!h || !sums_dev) return fail(DTFILL_E_ARG, "dtfill_eval_totals: NULL handle or sums");
    CU(cudaSetDevice(h->device));
    int rc = dtfill_flush(h);                 // the handle's stream now follows every call in flight
    if (rc) return rc;
    LaneTotals lt;
    for (int l = 0; l < dtfill_ctx::MAX_LANES; ++l)
        lt.p[l] = h->lanes[l].ev_dirty ? (const double*)h->lanes[l].ev_totals.p : nullptr;
    k4_fold_totals<<<1, 32, 0, h->stream>>>(lt, sums_dev, accumulate);
    for (Lane& L : h->lanes)
        if (L.ev_dirty) { CU(cudaMemsetAsync(L.ev_totals.p, 0, 10 * 8, h->stream)); L.ev_dirty = false; }
    CU(cudaGetLastError());
    return 0;
}

int dtfill_metrics(dtfill_t* h, const float* pred, const void* gt, int gt_is_f64, int in_is_device, int B, int H, int W,
                   int mode, double* per_frame, double* sums, int out_is_device) {
    return dtfill_metrics_ex(h, pred, gt, gt_is_f64, in_is_device, B, H, W, mode, per_frame, sums, out_is_device, 0);
}

int dtfill_metrics_ex(dtfill_t* h, const float* pred, const void* gt, int gt_is_f64, int in_is_device, int B, int H, int W,
                      int mode, double* per_frame, double* sums, int out_is_device, int accumulate) {
    if (!h || !pred || !gt) return fail(DTFILL_E_ARG, "dtfill_metrics: NULL handle or input");
    if (accumulate && !(out_is_device && sums))
        return fail(DTFILL_E_ARG, "dtfill_metrics_ex: accumulate needs a device-resident sums vector");
    if (B <= 0 || H <= 0 || W <= 0) return fail(DTFILL_E_ARG, "dtfill_metrics: B, H, W must be positive");
    if (mode != DTFILL_METRICS_KITTI && mode != DTFILL_METRICS_NYU) return fail(DTFILL_E_ARG, "dtfill_metrics: bad mode");
    CU(cudaSetDevice(h->device));
    { int frc = dtfill_flush(h); if (frc) return frc; }      // pipelined fills feeding this evaluation
    const long npx = (long)H * W;
    const size_t tot = (size_t)B * npx;
    const size_t gsz = gt_is_f64 ? 8 : 4;
    int rc;
    const float* p_d = pred;
    const void* g_d = gt;
    cudaStream_t s = h->stream;
    if (!in_is_device) {
        if ((rc = ensure(h, h->in_dev, tot * 4))) return rc;
        if ((rc = ensure(h, h->gt_dev, tot * gsz))) return rc;
        CU(cudaMemcpyAsync(h->in_dev.p, pred, tot * 4, cudaMemcpyHostToDevice, s));
        CU(cudaMemcpyAsync(h->gt_dev.p, gt, tot * gsz, cudaMemcpyHostToDevice, s));
        p_d = (const float*)h->in_dev.p;
        g_d = h->gt_dev.p;
    }
    if ((rc = ensure(h, h->per_frame, (size_t)B * 9 * 8))) return rc;
    if ((rc = ensure(h, h->sums, 10 * 8))) return rc;
    double* pf_d = (out_is_device && per_frame) ? per_frame : (double*)h->per_frame.p;
    double* sm_d = (out_is_device && sums) ? sums : (double*)h->sums.p;
    if (h->metrics_exact && npx < (1l << 31)) {
        const double* g64 = (const double*)g_d;
        const float* g32 = (const float*)g_d;
        if (gt_is_f64)
            rc = mode == 0 ? k4x_enqueue<double, 0>(h, p_d, g64, B, npx, pf_d, s) : k4x_enqueue<double, 1>(h, p_d, g64, B, npx, pf_d, s);
        else
            rc = mode == 0 ? k4x_enqueue<float, 0>(h, p_d, g32, B, npx, pf_d, s) : k4x_enqueue<float, 1>(h, p_d, g32, B, npx, pf_d, s);
        if (rc) return rc;
        k4x_sums<<<1, 32, 0, s>>>(pf_d, B, sm_d, accumulate);
    } else {
    int chunks = (int)((npx + 16383) / 16384);     // chunk boundaries stay multiples of 4 pixels when npx is
    if (chunks < 1) chunks = 1;
    if (chunks > 64) chunks = 64;
    while (chunks > 1 && (((npx + chunks - 1) / chunks) & 3)) --chunks;
    if ((rc = ensure(h, h->partial, (size_t)B * chunks * ACC * 8))) return rc;
    dim3 grid(chunks, B);
    double* part = (double*)h->partial.p;
    if (gt_is_f64) {
        if (mode == 0) k4_metrics_partial<double, 0><<<grid, 256, 0, s>>>(p_d, (const double*)g_d, npx, chunks, part);
        else k4_metrics_partial<double, 1><<<grid, 256, 0, s>>>(p_d, (const double*)g_d, npx, chunks, part);
    } else {
        if (mode == 0) k4_metrics_partial<float, 0><<<grid, 256, 0, s>>>(p_d, (const float*)g_d, npx, chunks, part);
        else k4_metrics_partial<float, 1><<<grid, 256, 0, s>>>(p_d, (const float*)g_d, npx, chunks, part);
    }
    k4_metrics_final<<<1, 256, 0, s>>>(part, B, chunks, mode, pf_d, sm_d, accumulate);
    }
    CU(cudaGetLastError());
    if (!out_is_device) {
        if (per_frame) CU(cudaMemcpyAsync(per_frame, pf_d, (size_t)B * 9 * 8, cudaMemcpyDeviceToHost, s));
        if (sums) CU(cudaMemcpyAsync(sums, sm_d, 10 * 8, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
    }
    return 0;
}

int dtfill_eval_png(dtfill_t* h, const uint8_t* lidar, const int64_t* lidar_offsets, const uint8_t* gt,
                    const int64_t* gt_offsets, int B, int H, int W, float src_thr, float val_thr, double* per_frame,
                    double* sums, int* first_bad_frame) {
    if (first_bad_frame) *first_bad_frame = -1;
    if (!h || !lidar || !lidar_offsets || !gt || !gt_offsets)
        return fail(DTFILL_E_ARG, "dtfill_eval_png: NULL handle, files or offsets");
    if (B <= 0 || H <= 0 || W <= 0) return fail(DTFILL_E_ARG, "dtfill_eval_png: B, H, W must be positive");
    if ((int64_t)H * (1 + 2 * (int64_t)W) >= (1ll << 28))
        return fail(DTFILL_E_ARG, "dtfill_eval_png: frame too large (H * (1 + 2 W) < 2^28 bytes)");
    CU(cudaSetDevice(h->device));
    const long npx = (long)H * W;
    cudaStream_t s = h->stream;
    int rc;
    // 1. one decode of the 2B files (one warp per file, so the call costs about the slowest file, not two files in a row):
    //    LiDAR file b -> samples / status b, ground-truth file b -> samples / status B + b
    if ((rc = ensure(h, h->png_samples, (size_t)2 * B * npx * 2))) return rc;
    if ((rc = ensure(h, h->png_status, (size_t)2 * B * 4))) return rc;
    int32_t* st_host = nullptr;                   // [2B] decode status, then the fill's counts [B][2]
    if ((rc = png_status_host(h, 4 * B, &st_host))) return rc;
    uint16_t* samples = (uint16_t*)h->png_samples.p;
    int32_t* status = (int32_t*)h->png_status.p;
    const PngFiles sets[2] = {{lidar, lidar_offsets, B}, {gt, gt_offsets, B}};
    const uint8_t* d_data;
    const int64_t* d_off;
    if ((rc = png_stage(h, sets, 2, &d_data, &d_off))) return rc;
    const size_t h2d = h->last_h2d_bytes;
    if ((rc = png_enqueue(h, d_data, d_off, 1, 2 * B, H, W, samples, status))) return rc;
    // 2. the fill of dtfill_run_u16 (no crop) on the LiDAR samples, strict order on the handle's stream; only the counts
    //    leave the device
    if ((rc = ensure(h, h->depth_dev, (size_t)B * npx * 4))) return rc;
    if ((rc = ensure(h, h->counts_out_dev, (size_t)B * 8))) return rc;
    float* depth = (float*)h->depth_dev.p;
    int32_t* counts = (int32_t*)h->counts_out_dev.p;
    {
        InputScope scope(h, true, H, 0, nullptr);
        if ((rc = enqueue(h, samples, B, H, W, src_thr, val_thr, depth, nullptr, nullptr, nullptr, counts, nullptr, true)))
            return rc;
    }
    // 3. Result.evaluate of the filled depth against the ground-truth samples, in numpy's summation order whatever
    //    dtfill_set_metrics_exact says
    if ((rc = ensure(h, h->per_frame, (size_t)B * 9 * 8))) return rc;
    if ((rc = ensure(h, h->sums, 10 * 8))) return rc;
    double* pf_d = (double*)h->per_frame.p;
    double* sm_d = (double*)h->sums.p;
    if ((rc = k4x_enqueue<double, 0>(h, depth, samples + (size_t)B * npx, B, npx, pf_d, s))) return rc;
    k4x_sums<<<1, 32, 0, s>>>(pf_d, B, sm_d, 0);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(st_host, status, (size_t)2 * B * 4, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(st_host + 2 * B, counts, (size_t)B * 8, cudaMemcpyDeviceToHost, s));
    if (per_frame) CU(cudaMemcpyAsync(per_frame, pf_d, (size_t)B * 9 * 8, cudaMemcpyDeviceToHost, s));
    if (sums) CU(cudaMemcpyAsync(sums, sm_d, 10 * 8, cudaMemcpyDeviceToHost, s));
    int fill_bad = -1;
    rc = dtfill_status(h, &fill_bad, nullptr);       // synchronises
    h->last_h2d_bytes = h2d;
    h->last_d2h_bytes = (size_t)B * (2 * 4 + 8 + (per_frame ? 9 * 8 : 0)) + (sums ? 10 * 8 : 0);
    if (rc != 0 && rc != DTFILL_E_INDEX) return rc;
    // 4. the verdict, frame by frame as the notebook's loop meets it: a decode failure (LiDAR before ground truth) wins
    //    over an IndexError of Distance_Transform
    for (int b = 0; b < B; ++b) {
        const bool lid_bad = st_host[b] != png::ST_OK;
        if (lid_bad || st_host[B + b] != png::ST_OK) {
            const int st = lid_bad ? st_host[b] : st_host[B + b];
            if (first_bad_frame) *first_bad_frame = b;
            return fail(DTFILL_E_DATA, std::string(lid_bad ? "LiDAR" : "ground-truth") + " file " + std::to_string(b) + ": " +
                                           png_reason(st) + " (status " + std::to_string(st) + ")");
        }
    }
    return fill_verdict(rc, fill_bad, st_host + 2 * B, B, "LiDAR file ", first_bad_frame);
}

int dtfill_eval_sampled(dtfill_t* h, const float* gt, int gt_is_device, int B, int H, int W, const int32_t* rows,
                        const int32_t* cols, const int64_t* sample_offsets, int coords_are_device, int r0, int r1, int c0,
                        int c1, float src_thr, float val_thr, float* out_lidar, double* per_frame, double* sums,
                        int* first_bad_frame) {
    const char* who = "dtfill_eval_sampled";
    if (first_bad_frame) *first_bad_frame = -1;
    if (!h || !gt || !rows || !cols || !sample_offsets)
        return fail(DTFILL_E_ARG, std::string(who) + ": NULL handle, ground truth, coordinates or offsets");
    if (B <= 0 || H <= 0 || W <= 0) return fail(DTFILL_E_ARG, std::string(who) + ": B, H, W must be positive");
    if ((long)H + W >= 60000 || (long)H * W >= (1l << 31) || W > 28000)
        return fail(DTFILL_E_ARG, std::string(who) + ": frame size not supported (H + W < 60000, W <= 28000)");
    if (r0 < 0 || r1 > H || r0 >= r1 || c0 < 0 || c1 > W || c0 >= c1)
        return fail(DTFILL_E_ARG, std::string(who) + ": window [" + std::to_string(r0) + ":" + std::to_string(r1) + ", " +
                                      std::to_string(c0) + ":" + std::to_string(c1) + "] is not a non-empty window of the " +
                                      std::to_string(H) + " x " + std::to_string(W) + " frame");
    if (gt_is_device && (W & 3) == 0 && ((uintptr_t)gt & 15))
        return fail(DTFILL_E_ARG, std::string(who) + ": device ground truth must be 16-byte aligned");
    CU(cudaSetDevice(h->device));
    int rc = dtfill_flush(h);        // fills in flight (pipelined mode) may still use lane 0's workspace
    if (rc) return rc;
    const long npx = (long)H * W;
    const int WW = (W + 31) / 32;
    cudaStream_t s = h->stream;
    size_t h2d = 0;
    // 1. coordinates: host ones are checked here and go up in one copy through the pinned staging buffer (rows, cols, then
    //    the offsets rebased to 0); device ones are checked by k10_sample_bits
    const int32_t* d_rows = rows;
    const int32_t* d_cols = cols;
    const int64_t* d_off = sample_offsets;
    if (!coords_are_device) {
        const int64_t* o = sample_offsets;
        if (o[0] < 0) return fail(DTFILL_E_ARG, std::string(who) + ": sample_offsets[0] < 0");
        for (int b = 0; b < B; ++b) {
            if (o[b + 1] < o[b]) {
                if (first_bad_frame) *first_bad_frame = b;
                return fail(DTFILL_E_ARG, std::string(who) + ": frame " + std::to_string(b) + " has a negative sample count");
            }
            for (int64_t i = o[b]; i < o[b + 1]; ++i)
                if ((unsigned)rows[i] >= (unsigned)H || (unsigned)cols[i] >= (unsigned)W) {
                    if (first_bad_frame) *first_bad_frame = b;
                    return fail(DTFILL_E_ARG, std::string(who) + ": frame " + std::to_string(b) + ": sample (" +
                                                  std::to_string(rows[i]) + ", " + std::to_string(cols[i]) +
                                                  ") outside the frame");
                }
        }
        const size_t n = (size_t)(o[B] - o[0]);
        const size_t off_at = (2 * n * 4 + 15) & ~(size_t)15;
        const size_t total = off_at + (size_t)(B + 1) * 8;
        if ((rc = ensure_pinned(h->pin_smp, total))) return rc;
        if ((rc = ensure(h, h->smp_coords, total))) return rc;
        uint8_t* pin = (uint8_t*)h->pin_smp.p;
        if (n) {
            memcpy(pin, rows + o[0], n * 4);
            memcpy(pin + n * 4, cols + o[0], n * 4);
        }
        int64_t* po = (int64_t*)(pin + off_at);
        for (int b = 0; b <= B; ++b) po[b] = o[b] - o[0];
        CU(cudaMemcpyAsync(h->smp_coords.p, pin, total, cudaMemcpyHostToDevice, s));
        h2d += total;
        d_rows = (const int32_t*)h->smp_coords.p;
        d_cols = d_rows + n;
        d_off = (const int64_t*)((uint8_t*)h->smp_coords.p + off_at);
    }
    // 2. the ground truth, unless it is resident
    const float* g_d = gt;
    if (!gt_is_device) {
        if ((rc = ensure(h, h->gt_dev, (size_t)B * npx * 4))) return rc;
        CU(cudaMemcpyAsync(h->gt_dev.p, gt, (size_t)B * npx * 4, cudaMemcpyHostToDevice, s));
        h2d += (size_t)B * npx * 4;
        g_d = (const float*)h->gt_dev.p;
    }
    // 3. the sample bitmap in lane 0's srcbits (the lane of a strict-order fill), sized as the fill sizes it so that the
    //    fill does not reallocate it
    Lane* L = &h->lanes[0];
    if ((rc = ensure(h, L->srcbits, (size_t)B * H * WW * 4))) return rc;
    if ((rc = ensure(h, h->smp_bad, 4))) return rc;
    CU(cudaMemsetAsync(L->srcbits.p, 0, (size_t)B * H * WW * 4, s));
    CU(cudaMemsetAsync(h->smp_bad.p, 0x7F, 4, s));           // 0x7F7F7F7F: above every frame index
    k10_sample_bits<<<B, K10_THREADS, 0, s>>>(d_rows, d_cols, d_off, H, W, WW, (uint32_t*)L->srcbits.p, (int*)h->smp_bad.p);
    CU(cudaGetLastError());
    // 4. the fill with K1's sampled input kind, strict order on the handle's stream; the filled depth stays on the device
    if ((rc = ensure(h, h->depth_dev, (size_t)B * npx * 4))) return rc;
    if ((rc = ensure(h, h->counts_out_dev, (size_t)B * 8))) return rc;
    float* lid_d = nullptr;
    if (out_lidar) {
        if ((rc = ensure(h, h->lidar_out_dev, (size_t)B * npx * 4))) return rc;
        lid_d = (float*)h->lidar_out_dev.p;
    }
    float* depth = (float*)h->depth_dev.p;
    int32_t* counts = (int32_t*)h->counts_out_dev.p;
    {
        InputScope scope(h, false, H, 0, lid_d);
        h->in_sampled = true;
        rc = enqueue(h, g_d, B, H, W, src_thr, val_thr, depth, nullptr, nullptr, nullptr, counts, nullptr, true);
        h->in_sampled = false;
        if (rc) return rc;
    }
    // 5. Result_NYU.evaluate of the window of the filled depth against the same window of the ground truth, in numpy's
    //    summation order whatever dtfill_set_metrics_exact says
    if ((rc = ensure(h, h->per_frame, (size_t)B * 9 * 8))) return rc;
    if ((rc = ensure(h, h->sums, 10 * 8))) return rc;
    double* pf_d = (double*)h->per_frame.p;
    double* sm_d = (double*)h->sums.p;
    const K4xWindow win{npx, W, r0, c0, c1 - c0};
    if ((rc = k4x_enqueue<float, 1, float, true>(h, depth, g_d, B, (long)(r1 - r0) * (c1 - c0), pf_d, s, win))) return rc;
    k4x_sums<<<1, 32, 0, s>>>(pf_d, B, sm_d, 0);
    CU(cudaGetLastError());
    if ((rc = ensure_pinned(h->pin_smp_out, (size_t)B * 8 + 4))) return rc;
    int32_t* out_h = (int32_t*)h->pin_smp_out.p;            // the fill's counts [B][2], then the flag word
    CU(cudaMemcpyAsync(out_h, counts, (size_t)B * 8, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(out_h + 2 * B, h->smp_bad.p, 4, cudaMemcpyDeviceToHost, s));
    if (per_frame) CU(cudaMemcpyAsync(per_frame, pf_d, (size_t)B * 9 * 8, cudaMemcpyDeviceToHost, s));
    if (sums) CU(cudaMemcpyAsync(sums, sm_d, 10 * 8, cudaMemcpyDeviceToHost, s));
    if (out_lidar) CU(cudaMemcpyAsync(out_lidar, lid_d, (size_t)B * npx * 4, cudaMemcpyDeviceToHost, s));
    int fill_bad = -1;
    rc = dtfill_status(h, &fill_bad, nullptr);       // synchronises
    h->last_h2d_bytes = h2d;
    h->last_d2h_bytes = (size_t)B * 8 + 4 + (per_frame ? (size_t)B * 9 * 8 : 0) + (sums ? 10 * 8 : 0) +
                        (out_lidar ? (size_t)B * npx * 4 : 0);
    if (rc != 0 && rc != DTFILL_E_INDEX) return rc;
    // 6. the verdict: device coordinates outside the frame, then Distance_Transform's frame by frame
    const int bad = out_h[2 * B];
    if (bad < B) {
        if (first_bad_frame) *first_bad_frame = bad;
        return fail(DTFILL_E_ARG, std::string(who) + ": frame " + std::to_string(bad) +
                                      ": a sample outside the frame, or a negative sample count");
    }
    return fill_verdict(rc, fill_bad, out_h, B, "frame ", first_bad_frame);
}

int dtfill_set_band_cap(dtfill_t* h, int cap) {
    if (!h) return fail(DTFILL_E_ARG, "dtfill_set_band_cap: NULL handle");
    h->band_cap = cap;
    return 0;
}

int dtfill_set_sky_min(dtfill_t* h, int rows) {
    if (!h || rows < -1) return fail(DTFILL_E_ARG, "dtfill_set_sky_min: NULL handle or row count below -1");
    h->sky_min = rows;
    return 0;
}

int dtfill_debug_get_tasks(dtfill_t* h, int32_t* out, int max_tasks) {
    if (!h || !out || max_tasks < 0) return fail(DTFILL_E_ARG, "dtfill_debug_get_tasks: bad argument");
    static_assert(sizeof(Task) == 48, "Task layout is part of the debug ABI");
    CU(cudaSetDevice(h->device));
    { int rc = dtfill_synchronize(h); if (rc) return rc; }
    const Lane& L = h->lanes[h->last_lane];
    long n = (long)L.last_B * MAXT;
    if (n > max_tasks) n = max_tasks;
    if (n > 0) CU(cudaMemcpy(out, L.tasks.p, (size_t)n * sizeof(Task), cudaMemcpyDeviceToHost));
    return (int)n;
}

int dtfill_debug_read_status(dtfill_t* h, int32_t* out, int n) {
    if (!h || !out || n < 0 || n > 64) return fail(DTFILL_E_ARG, "dtfill_debug_read_status: bad argument");
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaMemcpy(out, h->status_dev + (size_t)h->last_slot * dtfill_ctx::STATUS_STRIDE, (size_t)n * 4, cudaMemcpyDeviceToHost));
    return 0;
}

#ifdef DTFILL_TRACE
// tuning build: (re)arm the trace buffer / read it back: out[calls][4 kernels][4] u64 = first start, last end, sum, blocks
extern "C" int dtfill_debug_trace_arm(dtfill_t* h) {
    CU(cudaSetDevice(h->device));
    const size_t n = (size_t)dtfill_ctx::TRACE_CALLS * 16;
    if (!h->trace_dev) CU(cudaMalloc(&h->trace_dev, n * 8));
    std::vector<unsigned long long> init(n);
    for (size_t i = 0; i < n; ++i) init[i] = (i % 4 == 0) ? ~0ull : 0ull;
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(h->trace_dev, init.data(), n * 8, cudaMemcpyHostToDevice));
    h->ncalls = 0;
    return 0;
}
extern "C" int dtfill_debug_trace_read(dtfill_t* h, unsigned long long* out) {
    CU(cudaSetDevice(h->device));
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(out, h->trace_dev, (size_t)dtfill_ctx::TRACE_CALLS * 16 * 8, cudaMemcpyDeviceToHost));
    return 0;
}
#endif

int dtfill_debug_set_skip(dtfill_t* h, int mask) {
    if (!h) return fail(DTFILL_E_ARG, "dtfill_debug_set_skip: NULL handle");
    h->debug_skip = mask;
    return 0;
}

int dtfill_set_subbatches(dtfill_t* h, int n) {
    if (!h) return fail(DTFILL_E_ARG, "dtfill_set_subbatches: NULL handle");
    h->nsub = n;
    return 0;
}

int dtfill_set_stage_threads(dtfill_t* h, int threads) {
    if (!h || threads < -1 || threads > 64) return fail(DTFILL_E_ARG, "dtfill_set_stage_threads: NULL handle or thread count outside -1..64");
    if (threads != h->stage_threads) {
        delete h->pool_in; delete h->pool_out;
        h->pool_in = h->pool_out = nullptr;
        h->stage_threads = threads;
    }
    return 0;
}

// Host-only hook for the CPU test-suite (no handle, no device): the compaction of the sparse upload on one block of pixels.
long dtfill_debug_compact(const float* src, long n, float src_thr, float val_thr, uint32_t* idx, uint32_t* val, long cap) {
    if (!src || !idx || !val || n < 0 || cap < n + (long)COMPACT_SLACK) return -1;      // the packed stores need slack
    return (long)compact_block(src, (size_t)n, 0u, source_cut(src_thr), val_thr, idx, val);
}

int dtfill_set_metrics_exact(dtfill_t* h, int enabled) {
    if (!h) return fail(DTFILL_E_ARG, "dtfill_set_metrics_exact: NULL handle");
    h->metrics_exact = enabled != 0;
    return 0;
}

int dtfill_set_sparse_upload(dtfill_t* h, int enabled) {
    if (!h) return fail(DTFILL_E_ARG, "dtfill_set_sparse_upload: NULL handle");
    h->sparse_upload = enabled != 0;
    return 0;
}

int dtfill_transfer_bytes(dtfill_t* h, unsigned long long* h2d, unsigned long long* d2h) {
    if (!h) return fail(DTFILL_E_ARG, "dtfill_transfer_bytes: NULL handle");
    if (h2d) *h2d = h->last_h2d_bytes;
    if (d2h) *d2h = h->last_d2h_bytes;
    return 0;
}

int dtfill_set_profiling(dtfill_t* h, int enabled) {
    if (!h) return fail(DTFILL_E_ARG, "dtfill_set_profiling: NULL handle");
    h->profiling = enabled != 0;
    return 0;
}

int dtfill_kernel_times(dtfill_t* h, float* ms) {
    if (!h || !ms) return fail(DTFILL_E_ARG, "dtfill_kernel_times: NULL argument");
    if (!h->profiling) return fail(DTFILL_E_ARG, "dtfill_kernel_times: profiling is off");
    CU(cudaSetDevice(h->device));
    CU(cudaEventSynchronize(h->ev[DTFILL_NUM_KERNELS]));
    for (int i = 0; i < DTFILL_NUM_KERNELS; ++i) CU(cudaEventElapsedTime(&ms[i], h->ev[i], h->ev[i + 1]));
    return 0;
}

int dtfill_dt_pool_ex(dtfill_t* h, const float* data, const float* mask, int in_is_device, int B, int H, int W,
                      int table_size, int scale_num, float* out, uint8_t* out_masks, int out_is_device) {
    if (!h || !data || !mask) return fail(DTFILL_E_ARG, "dtfill_dt_pool: NULL handle, data or mask");
    if (B <= 0 || H <= 0 || W <= 0) return fail(DTFILL_E_ARG, "dtfill_dt_pool: B, H, W must be positive");
    if (table_size < 1 || (table_size & 1) == 0 || table_size > 2 * K5_MAXR + 1)
        return fail(DTFILL_E_ARG, "dtfill_dt_pool: table_size must be odd and <= 15");       // net.py:72 assert
    if (scale_num < 1 || scale_num > 4) return fail(DTFILL_E_ARG, "dtfill_dt_pool: scale_num must be 1..4");
    if (scale_num == 1) return 0;
    if (!out) return fail(DTFILL_E_ARG, "dtfill_dt_pool: NULL out");
    CU(cudaSetDevice(h->device));
    { int frc = dtfill_flush(h); if (frc) return frc; }
    const size_t npx = (size_t)B * H * W;
    const int nl = scale_num - 1;
    cudaStream_t s = h->stream;
    int rc;
    const float* d_d = data; const float* m_d = mask; float* o_d = out;
    if (!in_is_device) {
        if ((rc = ensure(h, h->in_dev, npx * 4))) return rc;
        if ((rc = ensure(h, h->gt_dev, npx * 4))) return rc;
        CU(cudaMemcpyAsync(h->in_dev.p, data, npx * 4, cudaMemcpyHostToDevice, s));
        CU(cudaMemcpyAsync(h->gt_dev.p, mask, npx * 4, cudaMemcpyHostToDevice, s));
        d_d = (const float*)h->in_dev.p; m_d = (const float*)h->gt_dev.p;
    }
    uint8_t* k_d = out_masks;
    if (!out_is_device) {
        if ((rc = ensure(h, h->depth_dev, npx * 4 * nl))) return rc;
        o_d = (float*)h->depth_dev.p;
        if (out_masks) { if ((rc = ensure(h, h->mask_dev, npx * nl))) return rc; k_d = (uint8_t*)h->mask_dev.p; }
    }
    dim3 grid((W + K5_TW - 1) / K5_TW, (H + K5_TH - 1) / K5_TH, B);
    dim3 tgrid((W + 63) / 64, (H + 31) / 32, B);          // k5_dt_pool_tile: 64 x 32 outputs per block
    dim3 wgrid((W + 63) / 64, (H + 63) / 64, B);          // k5_dt_pool_win: 64 x 64 outputs per block
    for (int l = 0; l < nl; ++l) {
        const float* src = l == 0 ? d_d : o_d + (size_t)(l - 1) * npx;
        const float* msk = l == 0 ? m_d : nullptr;
        float* dst = o_d + (size_t)l * npx;
        uint8_t* dmk = k_d ? k_d + (size_t)l * npx : nullptr;
        const bool pvec = (W & 3) == 0 && ((uintptr_t)src & 15) == 0 && (!msk || ((uintptr_t)msk & 15) == 0);
        switch (table_size) {
            case 3: if (pvec) k5_dt_pool_win<1, true><<<wgrid, 256, 0, s>>>(src, msk, H, W, dst, dmk); else k5_dt_pool_win<1, false><<<wgrid, 256, 0, s>>>(src, msk, H, W, dst, dmk); break;
            case 5: if (pvec) k5_dt_pool_win<2, true><<<wgrid, 256, 0, s>>>(src, msk, H, W, dst, dmk); else k5_dt_pool_win<2, false><<<wgrid, 256, 0, s>>>(src, msk, H, W, dst, dmk); break;
            case 7: if (pvec) k5_dt_pool_win<3, true><<<wgrid, 256, 0, s>>>(src, msk, H, W, dst, dmk); else k5_dt_pool_win<3, false><<<wgrid, 256, 0, s>>>(src, msk, H, W, dst, dmk); break;
            case 9: k5_dt_pool_tile<4><<<tgrid, 256, 0, s>>>(src, msk, H, W, dst, dmk); break;
            default: k5_dt_pool_level<<<grid, 256, 0, s>>>(src, msk, H, W, table_size, dst, dmk); break;
        }
    }
    CU(cudaGetLastError());
    if (!out_is_device) {
        CU(cudaMemcpyAsync(out, o_d, npx * 4 * nl, cudaMemcpyDeviceToHost, s));
        if (out_masks) CU(cudaMemcpyAsync(out_masks, k_d, npx * nl, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
    }
    return 0;
}

int dtfill_dt_pool_demo(dtfill_t* h, const float* data, int in_is_device, int B, int H, int W, int table_size, int scale_num,
                        float* out, int out_is_device) {
    if (!h || !data) return fail(DTFILL_E_ARG, "dtfill_dt_pool_demo: NULL handle or data");
    if (B <= 0 || H <= 0 || W <= 0) return fail(DTFILL_E_ARG, "dtfill_dt_pool_demo: B, H, W must be positive");
    if (table_size < 1 || (table_size & 1) == 0 || table_size > 2 * K5_MAXR + 1)
        return fail(DTFILL_E_ARG, "dtfill_dt_pool_demo: table_size must be odd and <= 15");   // demo.py:66 assert
    if (scale_num < 1 || scale_num > 4) return fail(DTFILL_E_ARG, "dtfill_dt_pool_demo: scale_num must be 1..4");
    if (scale_num == 1) return 0;
    if (!out) return fail(DTFILL_E_ARG, "dtfill_dt_pool_demo: NULL out");
    CU(cudaSetDevice(h->device));
    { int frc = dtfill_flush(h); if (frc) return frc; }
    const size_t npx = (size_t)B * H * W;
    const int nl = scale_num - 1;
    cudaStream_t s = h->stream;
    int rc;
    const float* d_d = data; float* o_d = out;
    if (!in_is_device) {
        if ((rc = ensure(h, h->in_dev, npx * 4))) return rc;
        CU(cudaMemcpyAsync(h->in_dev.p, data, npx * 4, cudaMemcpyHostToDevice, s));
        d_d = (const float*)h->in_dev.p;
    }
    if (!out_is_device) {
        if ((rc = ensure(h, h->depth_dev, npx * 4 * nl))) return rc;
        o_d = (float*)h->depth_dev.p;
    }
    // demo.py:65-76: 10 ** (size - |i - middle| - |j - middle|) in float64, cast to float32
    float w[(2 * K5_MAXR + 1) * (2 * K5_MAXR + 1)];
    const int mid = (table_size - 1) / 2;
    for (int i = 0; i < table_size; ++i)
        for (int j = 0; j < table_size; ++j) {
            double p = 1.0;
            for (int k = 0; k < table_size - abs(i - mid) - abs(j - mid); ++k) p *= 10.0;      // exact in float64 (<= 1e15)
            w[i * table_size + j] = (float)p;
        }
    if ((rc = ensure(h, h->sums, 1024))) return rc;
    CU(cudaMemcpyAsync(h->sums.p, w, sizeof(float) * table_size * table_size, cudaMemcpyHostToDevice, s));
    CU(cudaStreamSynchronize(s));                     // w lives on this stack frame
    dim3 grid((W + K5_TW - 1) / K5_TW, (H + K5_TH - 1) / K5_TH, B);
    for (int l = 0; l < nl; ++l) {
        const float* src = l == 0 ? d_d : o_d + (size_t)(l - 1) * npx;
        k5_dt_pool_demo<<<grid, 256, 0, s>>>(src, (const float*)h->sums.p, H, W, table_size, o_d + (size_t)l * npx);
    }
    CU(cudaGetLastError());
    if (!out_is_device) {
        CU(cudaMemcpyAsync(out, o_d, npx * 4 * nl, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
    }
    return 0;
}

int dtfill_dt_pool(dtfill_t* h, const float* data, const float* mask, int in_is_device, int B, int H, int W,
                   int table_size, int scale_num, float* out, int out_is_device) {
    return dtfill_dt_pool_ex(h, data, mask, in_is_device, B, H, W, table_size, scale_num, out, nullptr, out_is_device);
}

int dtfill_outlier_removal(dtfill_t* h, const float* in, int in_is_device, int B, int H, int W, float* out,
                           int out_is_device) {
    if (!h || !in || !out) return fail(DTFILL_E_ARG, "dtfill_outlier_removal: NULL argument");
    if (B <= 0 || H <= 0 || W <= 0) return fail(DTFILL_E_ARG, "dtfill_outlier_removal: B, H, W must be positive");
    CU(cudaSetDevice(h->device));
    { int frc = dtfill_flush(h); if (frc) return frc; }
    const size_t npx = (size_t)B * H * W;
    cudaStream_t s = h->stream;
    int rc;
    const float* i_d = in; float* o_d = out;
    if (!in_is_device) {
        if ((rc = ensure(h, h->in_dev, npx * 4))) return rc;
        CU(cudaMemcpyAsync(h->in_dev.p, in, npx * 4, cudaMemcpyHostToDevice, s));
        i_d = (const float*)h->in_dev.p;
    }
    if (!out_is_device) {
        if ((rc = ensure(h, h->depth_dev, npx * 4))) return rc;
        o_d = (float*)h->depth_dev.p;
    }
    if (i_d == o_d) return fail(DTFILL_E_ARG, "dtfill_outlier_removal: out must not alias in (neighbours are read)");
    const bool vec = (W & 3) == 0 && ((uintptr_t)i_d & 15) == 0 && ((uintptr_t)o_d & 15) == 0;
    const long ngroups = vec ? (long)(npx / 4) : (long)npx;
    const unsigned grid = (unsigned)((ngroups + 255) / 256);
    if (vec) k6_outlier_removal<true><<<grid, 256, 0, s>>>(i_d, H, W, ngroups, o_d);
    else k6_outlier_removal<false><<<grid, 256, 0, s>>>(i_d, H, W, ngroups, o_d);
    CU(cudaGetLastError());
    if (!out_is_device) {
        CU(cudaMemcpyAsync(out, o_d, npx * 4, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
    }
    return 0;
}

int dtfill_edt(dtfill_t* h, const float* in, int in_is_device, int B, int H, int W, float src_thr, int32_t* out_d2,
               int32_t* out_idx, int out_is_device) {
    if (!h || !in || !out_d2) return fail(DTFILL_E_ARG, "dtfill_edt: NULL handle, input or out_d2");
    if (B <= 0 || H <= 0 || W <= 0) return fail(DTFILL_E_ARG, "dtfill_edt: B, H, W must be positive");
    if (H > 4096 || W > 25600)
        return fail(DTFILL_E_ARG, "dtfill_edt: frame size not supported (H <= 4096, W <= 25600)");
    CU(cudaSetDevice(h->device));
    { int frc = dtfill_flush(h); if (frc) return frc; }
    const size_t npx = (size_t)B * H * W;
    cudaStream_t s = h->stream;
    int rc;
    const float* i_d = in;
    if (!in_is_device) {
        if ((rc = ensure(h, h->in_dev, npx * 4))) return rc;
        CU(cudaMemcpyAsync(h->in_dev.p, in, npx * 4, cudaMemcpyHostToDevice, s));
        i_d = (const float*)h->in_dev.p;
    }
    int32_t* d2 = out_d2; int32_t* ix = out_idx;
    if (!out_is_device) {
        if ((rc = ensure(h, h->depth_dev, npx * 4))) return rc;
        d2 = (int32_t*)h->depth_dev.p;
        if (out_idx) { if ((rc = ensure(h, h->lbl_dev, npx * 4))) return rc; ix = (int32_t*)h->lbl_dev.p; }
    }
    if ((rc = ensure(h, h->edt_rows, npx * 2))) return rc;      // nearest source column per pixel (u16)
    if ((rc = ensure(h, h->edt_stack, npx * 8))) return rc;      // envelope stacks [frame][depth][column], 8 bytes per entry
    const long nrows = (long)B * H;
    {
        const unsigned grid = (unsigned)((nrows + 3) / 4);      // one warp per row
        if ((W & 7) == 0) k7_edt_rows<true><<<grid, 128, 0, s>>>(i_d, nrows, W, source_cut(src_thr), (uint16_t*)h->edt_rows.p);
        else k7_edt_rows<false><<<grid, 128, 0, s>>>(i_d, nrows, W, source_cut(src_thr), (uint16_t*)h->edt_rows.p);
    }
    // two scanlines per thread (the same column of frames b and b + B/2): see the kernel
    if (B >= 2) k7_edt_columns<2><<<dim3((W + 127) / 128, (B + 1) / 2), 128, 0, s>>>((const uint16_t*)h->edt_rows.p, B, H, W, (uint2*)h->edt_stack.p, d2, ix);
    else k7_edt_columns<1><<<dim3((W + 127) / 128, B), 128, 0, s>>>((const uint16_t*)h->edt_rows.p, B, H, W, (uint2*)h->edt_stack.p, d2, ix);
    CU(cudaGetLastError());
    if (!out_is_device) {
        CU(cudaMemcpyAsync(out_d2, d2, npx * 4, cudaMemcpyDeviceToHost, s));
        if (out_idx) CU(cudaMemcpyAsync(out_idx, ix, npx * 4, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
    }
    return 0;
}

int dtfill_host_alloc(void** out_ptr, size_t bytes) {
    if (!out_ptr) return fail(DTFILL_E_ARG, "dtfill_host_alloc: NULL out_ptr");
    *out_ptr = nullptr;
    cudaError_t e = cudaHostAlloc(out_ptr, bytes ? bytes : 1, cudaHostAllocDefault);
    if (e != cudaSuccess) return fail(DTFILL_E_NOMEM, std::string("cudaHostAlloc: ") + cudaGetErrorString(e));
    return 0;
}

void dtfill_host_free(void* ptr) {
    if (ptr) cudaFreeHost(ptr);
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------------------
// The one collective of the path (SURVEY.md 8(e)): an NCCL sum all-reduce of the running metric totals, issued on
// the handle's stream right behind k4_metrics_final.  libnccl is resolved at run time (dlopen of "libnccl.so.2":
// the copy a host framework already loaded is found first), so the library itself has no link-time dependency.
// ------------------------------------------------------------------------------------------------------------
namespace {

struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(void*) = nullptr;
    int (*CommInitRank)(void**, int, /*ncclUniqueId by value: 128 bytes*/ struct Id128, int) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
struct Id128 { char b[128]; };
NcclApi g_nccl;
std::mutex g_nccl_mu;

int nccl_load() {
    std::lock_guard<std::mutex> lk(g_nccl_mu);
    if (g_nccl.lib) return 0;
    const char* names[] = {getenv("DTFILL_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    void* lib = nullptr;
    for (const char* n : names)
        if (n && *n && (lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL))) break;
    if (!lib) return fail(DTFILL_E_CUDA, std::string("dtfill: cannot load libnccl.so.2 (") + dlerror() + ")");
    g_nccl.GetUniqueId = (int (*)(void*))dlsym(lib, "ncclGetUniqueId");
    g_nccl.CommInitRank = (int (*)(void**, int, Id128, int))dlsym(lib, "ncclCommInitRank");
    g_nccl.CommDestroy = (int (*)(void*))dlsym(lib, "ncclCommDestroy");
    g_nccl.AllReduce = (int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t))dlsym(lib, "ncclAllReduce");
    g_nccl.GetErrorString = (const char* (*)(int))dlsym(lib, "ncclGetErrorString");
    if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.CommDestroy || !g_nccl.AllReduce)
        return fail(DTFILL_E_CUDA, "dtfill: libnccl lacks ncclGetUniqueId / ncclCommInitRank / ncclAllReduce");
    g_nccl.lib = lib;
    return 0;
}

int nccl_fail(const char* what, int rc) {
    return fail(DTFILL_E_CUDA, std::string(what) + ": " + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "NCCL error") +
                                   " (" + std::to_string(rc) + ")");
}

}  // namespace

extern "C" {

int dtfill_nccl_unique_id(void* out_id) {
    if (!out_id) return fail(DTFILL_E_ARG, "dtfill_nccl_unique_id: NULL out_id");
    int rc = nccl_load();
    if (rc) return rc;
    rc = g_nccl.GetUniqueId(out_id);
    return rc ? nccl_fail("ncclGetUniqueId", rc) : 0;
}

int dtfill_comm_create(dtfill_t* h, const void* id, int nranks, int rank, void** out_comm) {
    if (!h || !id || !out_comm || nranks < 1 || rank < 0 || rank >= nranks)
        return fail(DTFILL_E_ARG, "dtfill_comm_create: bad argument");
    *out_comm = nullptr;
    int rc = nccl_load();
    if (rc) return rc;
    CU(cudaSetDevice(h->device));
    Id128 u;
    memcpy(u.b, id, sizeof(u.b));
    rc = g_nccl.CommInitRank(out_comm, nranks, u, rank);
    return rc ? nccl_fail("ncclCommInitRank", rc) : 0;
}

int dtfill_comm_destroy(void* comm) {
    if (!comm) return 0;
    int rc = nccl_load();
    if (rc) return rc;
    rc = g_nccl.CommDestroy(comm);
    return rc ? nccl_fail("ncclCommDestroy", rc) : 0;
}

int dtfill_allreduce_sums(dtfill_t* h, void* nccl_comm, double* sums_dev, int n) {
    if (!h || !nccl_comm || !sums_dev || n <= 0) return fail(DTFILL_E_ARG, "dtfill_allreduce_sums: bad argument");
    int rc = nccl_load();
    if (rc) return rc;
    CU(cudaSetDevice(h->device));
    if ((rc = dtfill_flush(h))) return rc;
    // in place, float64 sum, on the stream the metric kernels ran on: stream order is the only synchronisation
    rc = g_nccl.AllReduce(sums_dev, sums_dev, (size_t)n, /*ncclFloat64*/ 8, /*ncclSum*/ 0, nccl_comm, h->stream);
    return rc ? nccl_fail("ncclAllReduce", rc) : 0;
}

}  // extern "C"
