// dtfill_k11_draw.cuh -- K11: the NYU sample coordinates of a batch drawn on the device with numpy's legacy generator
// (RandomState, MT19937), the step before K10 of dtfill_eval_sampled_mt
#pragma once
#include "dtfill_common.cuh"

namespace dtfill {

// ------------------------------------------------------------------------------------------------------
// MT19937 as numpy's RandomState runs it.  The state is a 624-word key and pos; a word is taken as
//     if (pos == 624) { twist the key; pos = 0; }   y = temper(key[pos++])
// so the key is twisted lazily, only when a word is needed.  Over the whole stream, the raw (untempered) words form one
// sequence x with x[0..623] the key and block k+1 = twist(block k); word j of a draw that starts at pos is temper(x[pos + j]).
// RandomState.randint(k, size=n) (int64, k - 1 < 2^32 - 1) is masked rejection: with mask the smallest 2^j - 1 >= k - 1,
// each value is the first word v with (v & mask) <= k - 1, and the value is v & mask; k == 1 gives zeros and takes no word.
// ------------------------------------------------------------------------------------------------------
constexpr int MT_N = 624, MT_M = 397;

// One element of a twist: the new word from old[i] (upper bit), old[i+1] (lower bits) and the word 397 ahead (old) or 227
// behind (new).
__host__ __device__ __forceinline__ uint32_t mt_twist1(uint32_t hi, uint32_t lo, uint32_t far) {
    const uint32_t y = (hi & 0x80000000u) | (lo & 0x7fffffffu);
    return far ^ (y >> 1) ^ ((0u - (y & 1u)) & 0x9908b0dfu);
}

// Element i of the block that follows `o`, given the elements of that new block `d` computed so far.  Element i depends
// on new element i - 227 (i >= 227) and element 623 on new elements 0 and 396, so a block is three dependent stages:
// [0, 227), [227, 454), [454, 624).
__host__ __device__ __forceinline__ uint32_t mt_twist_elem(const uint32_t* o, const uint32_t* d, int i) {
    const uint32_t lo = i < MT_N - 1 ? o[i + 1] : d[0];
    const uint32_t far = i < MT_N - MT_M ? o[i + MT_M] : d[i - (MT_N - MT_M)];
    return mt_twist1(o[i], lo, far);
}

__host__ __device__ __forceinline__ void mt_twist_block(const uint32_t* o, uint32_t* d) {
    for (int i = 0; i < MT_N; ++i) d[i] = mt_twist_elem(o, d, i);
}

__host__ __device__ __forceinline__ uint32_t mt_temper(uint32_t y) {
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    return y ^ (y >> 18);
}

// numpy's gen_mask: the smallest 2^j - 1 >= rng
__host__ __device__ __forceinline__ uint32_t mt_mask(uint32_t rng) {
    rng |= rng >> 1; rng |= rng >> 2; rng |= rng >> 4; rng |= rng >> 8; rng |= rng >> 16;
    return rng;
}

// ------------------------------------------------------------------------------------------------------
// The draws of B frames as data_read.py:360-364 makes them, one frame after the other from one stream:
//     rows_b = randint(H - 12, size=n) + 6;  cols_b = randint(W - 16, size=n) + 8
// Phase 2b draws frame b's rows, phase 2b+1 its columns; each ends at its n-th accepted word.  A phase of range 1 takes no
// word (its values are the constant offset).  One block of K11_THREADS:
//   * generator warps (K11_GEN_THREADS) twist the next K11_G key blocks into one half of a shared double buffer, three
//     stages per block behind a named barrier, while
//   * the other warps take the half twisted before: temper every word and form both accept flags (row and column, 16 bits
//     each of one word), an inclusive block-wide prefix sum of the flags, and for each kind the index of its j-th accept
//     (a select table).  One thread then walks the phase boundaries: the end of the current phase is the select table's
//     entry at (accepts before the phase) + (accepts still needed), so each boundary costs two dependent shared loads.
//     It records where each phase starts in the half.  Last, every accepted word finds its phase by a binary search of
//     those starts and writes its value to its slot.
// Outputs: rows / cols int32 [B*n] (6 and 8 added), offsets int64 [B+1] = b*n, words int64 [B] (32-bit words frame b
// consumed), and the state numpy's lazy twist leaves: the key of the block that holds the last consumed word and pos just
// past it (624 is a valid pos); the input state itself when no word is consumed.
// ------------------------------------------------------------------------------------------------------
constexpr int K11_THREADS = 1024;
constexpr int K11_GEN_THREADS = 256;                       // warps 0..7 twist
constexpr int K11_USE_THREADS = K11_THREADS - K11_GEN_THREADS;
constexpr int K11_USE_WARPS = K11_USE_THREADS / 32;
constexpr int K11_G = 8;                                   // key blocks per half of the double buffer
constexpr int K11_S = K11_G * MT_N;                        // words per half: counts fit the 16-bit halves of a flag word
constexpr int K11_C = (K11_S + K11_USE_THREADS - 1) / K11_USE_THREADS;   // words per consumer thread
constexpr size_t K11_SMEM = (size_t)2 * K11_S * 4 /* raw */ + (size_t)K11_S * 4 /* prefix */ +
                            (size_t)2 * K11_S * 2 /* select */ + (size_t)(K11_S + 2) * 2 /* phase starts */;
static_assert(K11_S < 65536, "per-half accept counts are 16-bit");

__device__ __forceinline__ void k11_bar(int id, int count) {
    asm volatile("bar.sync %0, %1;" :: "r"(id), "r"(count) : "memory");
}

// The draws of one generator by one block: the body of k11_mt_draw and of each block of k11_mt_draw_many.  rows / cols
// point at the generator's first slot; offsets[b] = off_base + b * n for b < B, and for b == B too when write_end.
__device__ __forceinline__ void k11_draw(const uint32_t* __restrict__ key_in, int pos, int B, int n, uint32_t rng_r,
                                         uint32_t rng_c, int32_t* __restrict__ rows, int32_t* __restrict__ cols,
                                         int64_t* __restrict__ offsets, long long off_base, bool write_end,
                                         int64_t* __restrict__ words, uint32_t* __restrict__ key_out, int* __restrict__ pos_out)
{
    extern __shared__ __align__(16) uint8_t k11_smem[];
    uint32_t* raw = (uint32_t*)k11_smem;                      // [2][K11_S]
    uint32_t* P = raw + 2 * K11_S;                            // [K11_S] inclusive prefix of the packed flags
    uint16_t* sel = (uint16_t*)(P + K11_S);                   // [2][K11_S] index of the j-th accept, rows then cols
    uint16_t* seg = sel + 2 * K11_S;                          // [K11_S + 2] start of each phase in the half
    __shared__ uint32_t wsum[K11_USE_WARPS];
    __shared__ int nseg_s, p0_s, carry_s, done_s;
    __shared__ long long last_s;

    const int tid = threadIdx.x;
    const int nr = rng_r ? n : 0, nc = rng_c ? n : 0;        // words-consuming accepts per row / column phase
    const long long total = (long long)B * n;
    for (int b = tid; b < B + (int)write_end; b += K11_THREADS) offsets[b] = off_base + (long long)b * n;
    if (!rng_r) for (long long i = tid; i < total; i += K11_THREADS) rows[i] = 6;
    if (!rng_c) for (long long i = tid; i < total; i += K11_THREADS) cols[i] = 8;
    if (nr + nc == 0) {                                       // no word is consumed: the state comes back unchanged
        for (int b = tid; b < B; b += K11_THREADS) words[b] = 0;
        for (int i = tid; i < MT_N; i += K11_THREADS) key_out[i] = key_in[i];
        if (tid == 0) *pos_out = pos;
        return;
    }
    const uint32_t mr = mt_mask(rng_r), mc = mt_mask(rng_c);
    const int nph = 2 * B;
    // the walker's state (thread K11_GEN_THREADS), kept across halves
    int p = 0, have = 0;
    long long cur_e = pos, frame_start = pos;                 // next unconsumed word / first word of the current frame
    if (tid == K11_GEN_THREADS) {
        while (p < nph && ((p & 1) ? nc : nr) == 0) ++p;      // a leading row phase of range 1
        done_s = 0;
    }
    // half 0: block 0 is the key itself, blocks 1.. its twists
    if (tid < K11_GEN_THREADS) {
        for (int i = tid; i < MT_N; i += K11_GEN_THREADS) raw[i] = key_in[i];
        k11_bar(1, K11_GEN_THREADS);
        for (int g = 1; g < K11_G; ++g) {
            const uint32_t* o = raw + (g - 1) * MT_N;
            uint32_t* d = raw + g * MT_N;
            for (int st = 0; st < 3; ++st) {
                const int i = st * (MT_N - MT_M) + tid;
                if (tid < MT_N - MT_M && i < MT_N) d[i] = mt_twist_elem(o, d, i);
                k11_bar(1, K11_GEN_THREADS);
            }
        }
    }
    __syncthreads();
    const int ut = tid - K11_GEN_THREADS, lane = tid & 31, uw = ut >> 5;
    for (int k = 0;; ++k) {
        const int cur = k & 1;
        const long long base = (long long)k * K11_S;
        const uint32_t* buf = raw + cur * K11_S;
        if (tid < K11_GEN_THREADS) {
            // the next half, from the last block of this one
            uint32_t* nxt = raw + (cur ^ 1) * K11_S;
            for (int g = 0; g < K11_G; ++g) {
                const uint32_t* o = g ? nxt + (g - 1) * MT_N : buf + (K11_G - 1) * MT_N;
                uint32_t* d = nxt + g * MT_N;
                for (int st = 0; st < 3; ++st) {
                    const int i = st * (MT_N - MT_M) + tid;
                    if (tid < MT_N - MT_M && i < MT_N) d[i] = mt_twist_elem(o, d, i);
                    k11_bar(1, K11_GEN_THREADS);
                }
            }
        } else {
            // 1. flags: bit 0 a row accept, bit 16 a column accept; words before pos belong to no draw
            const int i0 = ut * K11_C;
            uint32_t f[K11_C];
            uint32_t run = 0;
#pragma unroll
            for (int j = 0; j < K11_C; ++j) {
                const int i = i0 + j;
                uint32_t a = 0;
                if (i < K11_S && base + i >= pos) {
                    const uint32_t v = mt_temper(buf[i]);
                    a = (uint32_t)(nr && (v & mr) <= rng_r) | ((uint32_t)(nc && (v & mc) <= rng_c) << 16);
                }
                run += a;
                f[j] = run;
            }
            // 2. block-wide inclusive prefix sum of the packed flags (no carry crosses the halves: counts < 2^16)
            uint32_t x = run;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, x, d);
                if (lane >= d) x += y;
            }
            if (lane == 31) wsum[uw] = x;
            k11_bar(2, K11_USE_THREADS);
            if (uw == 0) {
                uint32_t t = lane < K11_USE_WARPS ? wsum[lane] : 0;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t y = __shfl_up_sync(0xffffffffu, t, d);
                    if (lane >= d) t += y;
                }
                if (lane < K11_USE_WARPS) wsum[lane] = t;
            }
            k11_bar(2, K11_USE_THREADS);
            const uint32_t off = (uw ? wsum[uw - 1] : 0u) + x - run;
#pragma unroll
            for (int j = 0; j < K11_C; ++j) {
                const int i = i0 + j;
                if (i < K11_S) {
                    const uint32_t pi = off + f[j];
                    const uint32_t a = f[j] - (j ? f[j - 1] : 0u);
                    P[i] = pi;
                    if (a & 0xffffu) sel[(pi & 0xffffu) - 1] = (uint16_t)i;
                    if (a >> 16) sel[K11_S + (pi >> 16) - 1] = (uint16_t)i;
                }
            }
            k11_bar(2, K11_USE_THREADS);
            // 3. the phase boundaries, walked by one thread
            if (ut == 0) {
                int nseg = 0;
                int s = cur_e > base ? (int)(cur_e - base) : 0;       // where phase p starts in this half
                p0_s = p;
                carry_s = have;
                const uint32_t tot = P[K11_S - 1];
                while (p < nph) {
                    const int kind = p & 1;
                    const int sh = kind ? 16 : 0;
                    seg[nseg++] = (uint16_t)s;
                    const int before = s ? (int)((P[s - 1] >> sh) & 0xffffu) : 0;
                    const int avail = (int)((tot >> sh) & 0xffffu) - before;
                    const int need = n - have;
                    if (need > avail) { have += avail; break; }
                    const int i = sel[kind * K11_S + before + need - 1];
                    cur_e = base + i + 1;
                    s = i + 1;
                    have = 0;
                    do {                                               // and the phases of range 1 that follow it
                        if (p & 1) { words[p >> 1] = cur_e - frame_start; frame_start = cur_e; }
                        ++p;
                    } while (p < nph && ((p & 1) ? nc : nr) == 0);
                }
                if (p == nph) {
                    seg[nseg++] = (uint16_t)s;       // words after the last boundary belong to no phase
                    done_s = 1;
                    last_s = cur_e - 1;
                }
                nseg_s = nseg;
            }
            k11_bar(2, K11_USE_THREADS);
            // 4. every accepted word to its slot
            const int nseg = nseg_s, p0 = p0_s, carry = carry_s;
            const int step = (nr && nc) ? 1 : 2;                      // phases of range 1 have no segment
#pragma unroll
            for (int j = 0; j < K11_C; ++j) {
                const int i = i0 + j;
                const uint32_t a = f[j] - (j ? f[j - 1] : 0u);
                if (i >= K11_S || !a) continue;
                int lo = 0, hi = nseg - 1;                             // the last segment starting at or before i
                while (lo < hi) {
                    const int mid = (lo + hi + 1) >> 1;
                    if (seg[mid] <= i) lo = mid; else hi = mid - 1;
                }
                const int ph = p0 + lo * step;
                if (ph >= nph) continue;
                const int kind = ph & 1, sh = kind ? 16 : 0;
                if (!((a >> sh) & 1u)) continue;
                const int s0 = seg[lo];
                const int idx = (lo ? 0 : carry) + (int)(((off + f[j]) >> sh) & 0xffffu) -
                                (s0 ? (int)((P[s0 - 1] >> sh) & 0xffffu) : 0) - 1;
                const uint32_t v = mt_temper(buf[i]);
                const long long slot = (long long)(ph >> 1) * n + idx;
                if (kind) cols[slot] = (int32_t)(v & mc) + 8;
                else rows[slot] = (int32_t)(v & mr) + 6;
            }
            if (done_s) {
                const long long last = last_s;
                const uint32_t* blk = buf + (int)(last / MT_N - (long long)k * K11_G) * MT_N;
                for (int i = ut; i < MT_N; i += K11_USE_THREADS) key_out[i] = blk[i];
                if (ut == 0) *pos_out = (int)(last % MT_N) + 1;
            }
        }
        __syncthreads();
        if (done_s) break;
    }
}

__global__ void __launch_bounds__(K11_THREADS) k11_mt_draw(const uint32_t* __restrict__ key_in, int pos, int B, int n,
                                                          uint32_t rng_r, uint32_t rng_c, int32_t* __restrict__ rows,
                                                          int32_t* __restrict__ cols, int64_t* __restrict__ offsets,
                                                          int64_t* __restrict__ words, uint32_t* __restrict__ key_out,
                                                          int* __restrict__ pos_out)
{
    k11_draw(key_in, pos, B, n, rng_r, rng_c, rows, cols, offsets, 0, true, words, key_out, pos_out);
}

// D independent generators, one block each (dtfill_eval_sampled_mt_many): block d draws B frames of n_d samples from
// keys[d] / draws[d] = {pos_d, n_d}.  Its coordinates start at slot B * (n_0 + ... + n_{d-1}), its offsets are those of
// frames d*B .. d*B + B - 1 of the whole run (so k10_sample_bits reads the D*B frames as one batch; the last block writes
// offsets[D*B]), and its words, final key and pos go to row d of words [D][B], keys_out [D][624] and pos_out [D].
__global__ void __launch_bounds__(K11_THREADS) k11_mt_draw_many(const uint32_t* __restrict__ keys,
                                                               const int32_t* __restrict__ draws, int D, int B,
                                                               uint32_t rng_r, uint32_t rng_c, int32_t* __restrict__ rows,
                                                               int32_t* __restrict__ cols, int64_t* __restrict__ offsets,
                                                               int64_t* __restrict__ words, uint32_t* __restrict__ keys_out,
                                                               int* __restrict__ pos_out)
{
    const int d = blockIdx.x;
    long long base = 0;
    for (int e = 0; e < d; ++e) base += (long long)B * draws[2 * e + 1];
    k11_draw(keys + (size_t)d * MT_N, draws[2 * d], B, draws[2 * d + 1], rng_r, rng_c, rows + base, cols + base,
             offsets + (size_t)d * B, base, d == D - 1, words + (size_t)d * B, keys_out + (size_t)d * MT_N, pos_out + d);
}

}  // namespace dtfill
