// dtfill_k9_png_encode.cuh -- batched encoder of 16-bit grayscale PNG files, the mirror of dtfill_k8_png.cuh: uint16
// samples (or float32 depth in metres) [B,H,W] on the device become B PNG files, so that filled depth maps leave the
// device as compressed bytes (KITTI's depth-completion submissions and cached DT_NN maps are such files).
//
// Output: colour type 0, bit depth 16, no interlace; signature, IHDR, an IDAT holding the 2-byte zlib header, one IDAT
// per segment of SEG_ROWS rows, an IDAT holding the Adler-32, IEND.  The bytes are a pure function of the samples:
// dtfill_debug_png_encode_host runs the same definitions serially on the CPU and writes identical files.
//
//   k9_png_filter   one warp per row: the five filtered rows in PNG's big-endian byte order, the one with the least sum
//                   of absolute signed differences (libpng's heuristic; ties to the lowest type), filter byte + row
//                   into the frame's scratch of H*(1+2W) bytes, and the row's Adler-32.
//   k9_png_deflate  one warp per segment.  At every position p the walk takes the longest of four candidates, each
//                   verified byte by byte (ties to the smallest distance): distance 1, distance 2, one row back
//                   (1+2W), and the latest q in [segment start, p) with the same 3-byte hash.  The fixed distances may
//                   reach into the previous segment (the decoder is sequential); the hash candidate stays inside the
//                   segment; no match runs past the segment's end.  Greedy parse, fixed Huffman codes, then an empty
//                   stored block (zlib's Z_SYNC_FLUSH) so that the segment ends byte aligned; the last segment's
//                   empty block carries BFINAL.  A segment whose coded size would exceed its stored size is written
//                   as stored blocks.  The warp writes the segment's IDAT chunk and its CRC-32.
//   k9_png_offsets  exclusive scan of the file sizes -> out_offsets [B+1].
//   k9_png_pack     the files back to back: header, segment chunks, Adler-32 chunk (combined from the rows'), IEND.
//
// Parallel parts of the deflate warp: the hash table (latest position per hash, in shared memory) is updated 32
// positions at a time and __match_any_sync gives each position its predecessor inside the step, so the candidate does
// not depend on the schedule; the four match lengths are found 32 bytes per step with ballots; 32 tokens at a time are
// coded by the lanes, their bit offsets come from a warp prefix sum, and the lanes OR their codes into a ring of words
// in shared memory.  Only the step p -> p + len is serial.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace dtfill {
namespace png {

constexpr int SEG_ROWS = 16;          // rows per segment (one IDAT chunk each)
constexpr int HBITS = 12;             // bits of the 3-byte hash
constexpr int HSIZE = 1 << HBITS;
constexpr uint32_t NO_POS = 0xffffffffu;
constexpr int WINDOW = 32768;
constexpr int MAX_MATCH = 258;
constexpr int STORED_MAX = 65535;     // bytes of one stored block
constexpr int RING = 64;              // words of the deflate warp's bit ring (a batch of 32 tokens adds <= 31)
constexpr int HEAD_BYTES = 8 + 25 + 14;     // signature, IHDR, IDAT with the zlib header
constexpr int TAIL_BYTES = 16 + 12;         // IDAT with the Adler-32, IEND
constexpr uint32_t CRC_POLY = 0xedb88320u;

// ---- samples and filters -------------------------------------------------------------------------------------------

// float32 depth in metres -> sample: clip(nan_to_num(fl32(d * 256), nan=0, posinf=65535), 0, 65535) truncated toward
// zero.  Equals (d * 256).astype(np.uint16) for d in [0, 65535/256] and is the identity on d = k/256.
PNG_HD uint32_t depth_sample(float d) {
    const float v = d * 256.0f;
    if (!(v > 0.0f)) return 0;                    // NaN, zeros, negatives
    if (v >= 65535.0f) return 65535;              // +inf included
    return (uint32_t)v;
}

PNG_HD uint32_t filter_byte(int ft, uint32_t x, uint32_t a, uint32_t b, uint32_t c) {
    switch (ft) {
        case 1: return (x - a) & 255;
        case 2: return (x - b) & 255;
        case 3: return (x - ((a + b) >> 1)) & 255;
        case 4: return (x - (uint32_t)paeth((int)a, (int)b, (int)c)) & 255;
        default: return x;
    }
}

PNG_HD uint32_t msad(uint32_t v) { return v < 128 ? v : 256 - v; }

// Both filtered bytes of a sample (hi << 8 | lo) from the sample x and its neighbours a (left), b (above), c (above-left)
PNG_HD uint32_t filter_sample(int ft, uint32_t x, uint32_t a, uint32_t b, uint32_t c) {
    return (filter_byte(ft, x >> 8, a >> 8, b >> 8, c >> 8) << 8) | filter_byte(ft, x & 255, a & 255, b & 255, c & 255);
}

// ---- checksums ------------------------------------------------------------------------------------------------------

PNG_HD uint32_t crc_table_entry(uint32_t i) {
    uint32_t c = i;
    for (int k = 0; k < 8; ++k) c = (c & 1) ? (c >> 1) ^ CRC_POLY : c >> 1;
    return c;
}

// CRC-32 (PNG, zlib) of n bytes appended to a message whose CRC is crc
PNG_HD uint32_t crc32_bytes(const uint32_t* tab, uint32_t crc, const uint8_t* p, int64_t n) {
    uint32_t c = ~crc;
    for (int64_t i = 0; i < n; ++i) c = tab[(c ^ p[i]) & 255] ^ (c >> 8);
    return ~c;
}

// a(x) * b(x) mod P(x), bit-reflected (zlib's multmodp)
PNG_HD uint32_t multmodp(uint32_t a, uint32_t b) {
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        m >>= 1;
        b = (b & 1) ? (b >> 1) ^ CRC_POLY : b >> 1;
    }
    return p;
}

// CRC-32 of A || B from crc(A), crc(B) and len(B) (zlib's crc32_combine): crc(A) * x^(8 len2) + crc(B)
PNG_HD uint32_t crc32_combine(uint32_t crc1, uint32_t crc2, uint64_t len2) {
    uint32_t p = 1u << 31, sq = 1u << 23;         // x^0, x^8
    for (uint64_t n = len2; n; n >>= 1) {
        if (n & 1) p = multmodp(sq, p);
        sq = multmodp(sq, sq);
    }
    return multmodp(p, crc1) ^ crc2;
}

// Adler-32 of A || B from adler(A), adler(B) and len(B) (zlib's adler32_combine)
PNG_HD uint32_t adler32_combine(uint32_t adler1, uint32_t adler2, uint64_t len2) {
    const uint32_t rem = (uint32_t)(len2 % ADLER_MOD);
    uint32_t sum1 = adler1 & 0xffff;
    uint32_t sum2 = (uint32_t)(((uint64_t)rem * sum1) % ADLER_MOD);
    sum1 += (adler2 & 0xffff) + ADLER_MOD - 1;
    sum2 += ((adler1 >> 16) & 0xffff) + ((adler2 >> 16) & 0xffff) + ADLER_MOD - rem;
    if (sum1 >= ADLER_MOD) sum1 -= ADLER_MOD;
    if (sum1 >= ADLER_MOD) sum1 -= ADLER_MOD;
    if (sum2 >= 2 * ADLER_MOD) sum2 -= 2 * ADLER_MOD;
    if (sum2 >= ADLER_MOD) sum2 -= ADLER_MOD;
    return sum1 | (sum2 << 16);
}

PNG_HD void put_be32(uint8_t* p, uint32_t v) {
    p[0] = (uint8_t)(v >> 24); p[1] = (uint8_t)(v >> 16); p[2] = (uint8_t)(v >> 8); p[3] = (uint8_t)v;
}

// signature, IHDR chunk, IDAT chunk holding the zlib header 78 01 (32 KB window, no dictionary): HEAD_BYTES
PNG_HD void write_head(uint8_t* o, const uint32_t* tab, int H, int W) {
    const uint8_t sig[8] = {137, 80, 78, 71, 13, 10, 26, 10};
    for (int i = 0; i < 8; ++i) o[i] = sig[i];
    put_be32(o + 8, 13);
    put_be32(o + 12, T_IHDR);
    put_be32(o + 16, (uint32_t)W);
    put_be32(o + 20, (uint32_t)H);
    o[24] = 16; o[25] = 0; o[26] = 0; o[27] = 0; o[28] = 0;
    put_be32(o + 29, crc32_bytes(tab, 0, o + 12, 17));
    put_be32(o + 33, 2);
    put_be32(o + 37, T_IDAT);
    o[41] = 0x78; o[42] = 0x01;
    put_be32(o + 43, crc32_bytes(tab, 0, o + 37, 6));
}

// IDAT chunk holding the Adler-32, IEND: TAIL_BYTES
PNG_HD void write_tail(uint8_t* o, const uint32_t* tab, uint32_t adler) {
    put_be32(o, 4);
    put_be32(o + 4, T_IDAT);
    put_be32(o + 8, adler);
    put_be32(o + 12, crc32_bytes(tab, 0, o + 4, 8));
    put_be32(o + 16, 0);
    put_be32(o + 20, T_IEND);
    put_be32(o + 24, crc32_bytes(tab, 0, o + 20, 4));
}

// ---- DEFLATE --------------------------------------------------------------------------------------------------------

// Bytes of n bytes as stored blocks followed by the empty stored block of the sync flush
PNG_HD int64_t stored_bytes(int64_t n) { return n + 5 * ((n + STORED_MAX - 1) / STORED_MAX) + 5; }

PNG_HD int segments(int H) { return (H + SEG_ROWS - 1) / SEG_ROWS; }

// Worst-case size of one file: every segment stored, plus all chunk overhead
PNG_HD int64_t encode_bound(int H, int W) {
    const int64_t stride = 1 + 2 * (int64_t)W;
    int64_t n = HEAD_BYTES + TAIL_BYTES;
    for (int s = 0; s < segments(H); ++s) {
        const int rows = (H - s * SEG_ROWS) < SEG_ROWS ? H - s * SEG_ROWS : SEG_ROWS;
        n += 12 + stored_bytes(rows * stride);
    }
    return n;
}

PNG_HD uint32_t hash3(const uint8_t* f) {
    const uint32_t k = (uint32_t)f[0] | ((uint32_t)f[1] << 8) | ((uint32_t)f[2] << 16);
    return (k * 2654435761u) >> (32 - HBITS);
}

PNG_HD uint32_t bit_reverse(uint32_t v, int n) {
    uint32_t r = 0;
    for (int i = 0; i < n; ++i) r |= ((v >> i) & 1) << (n - 1 - i);
    return r;
}

// Fixed-Huffman bits of one token, LSB first: a literal (len < 3, val = byte) or a match (len 3..258, val = distance).
// Returns the number of bits (<= 31).
PNG_HD int token_bits(uint32_t len, uint32_t val, uint32_t* bits) {
    static constexpr uint16_t lbase[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59,
                                           67, 83, 99, 115, 131, 163, 195, 227, 258};
    static constexpr uint8_t lext[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
    static constexpr uint16_t dbase[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769,
                                           1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
    static constexpr uint8_t dext[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11,
                                         11, 12, 12, 13, 13};
    if (len < 3) {
        if (val < 144) { *bits = bit_reverse(0x30 + val, 8); return 8; }
        *bits = bit_reverse(0x190 + val - 144, 9);
        return 9;
    }
    int li = 28;
    while (lbase[li] > len) --li;
    const uint32_t sym = 257 + li;
    int n;
    uint32_t b;
    if (sym < 280) { b = bit_reverse(sym - 256, 7); n = 7; }
    else { b = bit_reverse(0xc0 + sym - 280, 8); n = 8; }
    b |= (len - lbase[li]) << n;
    n += lext[li];
    int di = 29;
    while (dbase[di] > val) --di;
    b |= bit_reverse((uint32_t)di, 5) << n;
    n += 5;
    b |= (val - dbase[di]) << n;
    n += dext[di];
    *bits = b;
    return n;
}

// Length of the match of f[p..] with f[p-d..], at most maxlen
PNG_HD int match_len(const uint8_t* f, int64_t p, int64_t d, int maxlen) {
    int n = 0;
    while (n < maxlen && f[p + n] == f[p - d + n]) ++n;
    return n;
}

// Segment s of a frame: filtered bytes [s0, s1)
PNG_HD void segment_range(int s, int H, int64_t stride, int64_t* s0, int64_t* s1) {
    const int r1 = (s + 1) * SEG_ROWS < H ? (s + 1) * SEG_ROWS : H;
    *s0 = (int64_t)s * SEG_ROWS * stride;
    *s1 = (int64_t)r1 * stride;
}

// Stored form of f[s0, s1): blocks of <= 65535 bytes, then the empty block (BFINAL when final).  Returns the size.
PNG_HD int64_t write_stored(const uint8_t* f, int64_t s0, int64_t s1, bool final_seg, uint8_t* o, int lane, int nlanes) {
    int64_t pos = 0;
    for (int64_t p = s0; p < s1; p += STORED_MAX) {
        const uint32_t n = (uint32_t)((s1 - p) < STORED_MAX ? s1 - p : STORED_MAX);
        if (lane == 0) {
            o[pos] = 0;
            o[pos + 1] = (uint8_t)n; o[pos + 2] = (uint8_t)(n >> 8);
            o[pos + 3] = (uint8_t)~n; o[pos + 4] = (uint8_t)(~n >> 8);
        }
        for (uint32_t i = lane; i < n; i += nlanes) o[pos + 5 + i] = f[p + i];
        pos += 5 + n;
    }
    if (lane == 0) {
        o[pos] = final_seg ? 1 : 0;
        o[pos + 1] = 0; o[pos + 2] = 0; o[pos + 3] = 0xff; o[pos + 4] = 0xff;
    }
    return pos + 5;
}

// ---- kernels --------------------------------------------------------------------------------------------------------

constexpr int K9_WARPS = 4;

// Row r of frame b, sample c, as a uint16 value (uint16 input, or float32 depth through depth_sample)
template <typename T>
__device__ __forceinline__ uint32_t load_sample(const T* row, int c);
template <>
__device__ __forceinline__ uint32_t load_sample<uint16_t>(const uint16_t* row, int c) { return row[c]; }
template <>
__device__ __forceinline__ uint32_t load_sample<float>(const float* row, int c) { return depth_sample(row[c]); }

// One warp per row: filter byte + filtered row into filt + b*H*(1+2W) + r*(1+2W), row_adler[b*H + r]
template <typename T>
__global__ void __launch_bounds__(32 * K9_WARPS) k9_png_filter(const T* __restrict__ in, int B, int H, int W,
                                                               uint8_t* __restrict__ filt, uint32_t* __restrict__ row_adler)
{
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t g = (int64_t)blockIdx.x * K9_WARPS + warp;
    if (g >= (int64_t)B * H) return;
    const int r = (int)(g % H);
    const int64_t stride = 1 + 2 * (int64_t)W;
    const T* x = in + g * W;
    const T* up = r ? x - W : nullptr;
    unsigned long long cost[5] = {0, 0, 0, 0, 0};
    for (int c = lane; c < W; c += 32) {
        const uint32_t v = load_sample(x, c), a = c ? load_sample(x, c - 1) : 0;
        const uint32_t bv = up ? load_sample(up, c) : 0, cv = (up && c) ? load_sample(up, c - 1) : 0;
#pragma unroll
        for (int ft = 0; ft < 5; ++ft) {
            const uint32_t y = filter_sample(ft, v, a, bv, cv);
            cost[ft] += msad(y >> 8) + msad(y & 255);
        }
    }
    int best = 0;
    unsigned long long best_cost = 0;
#pragma unroll
    for (int ft = 0; ft < 5; ++ft) {
        unsigned long long s = cost[ft];
        for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (ft == 0 || s < best_cost) { best = ft; best_cost = s; }
    }
    uint8_t* o = filt + g * stride;
    // Adler-32 of the row: a = 1 + sum x_i, b = n + sum (n - i) x_i over the n = 1 + 2W bytes (byte 0 the filter type)
    uint64_t sa = 0, sb = 0;
    for (int c = lane; c < W; c += 32) {
        const uint32_t v = load_sample(x, c), a = c ? load_sample(x, c - 1) : 0;
        const uint32_t bv = up ? load_sample(up, c) : 0, cv = (up && c) ? load_sample(up, c - 1) : 0;
        const uint32_t y = filter_sample(best, v, a, bv, cv);
        const uint32_t hi = y >> 8, lo = y & 255;
        o[1 + 2 * c] = (uint8_t)hi;
        o[2 + 2 * c] = (uint8_t)lo;
        sa += hi + lo;
        sb += (uint64_t)(stride - 1 - 2 * c) * hi + (uint64_t)(stride - 2 - 2 * c) * lo;
    }
    uint32_t a32 = (uint32_t)(sa % ADLER_MOD), b32 = (uint32_t)(sb % ADLER_MOD);
    for (int s = 16; s; s >>= 1) {
        a32 += __shfl_xor_sync(0xffffffffu, a32, s);
        b32 += __shfl_xor_sync(0xffffffffu, b32, s);
    }
    if (lane == 0) {
        o[0] = (uint8_t)best;
        const uint32_t A = (uint32_t)((1u + (uint64_t)a32 + (uint32_t)best) % ADLER_MOD);
        const uint32_t Bv = (uint32_t)(((uint64_t)stride % ADLER_MOD + b32 + (uint64_t)(stride % ADLER_MOD) * best) % ADLER_MOD);
        row_adler[g] = (Bv << 16) | A;
    }
}

struct DeflateSmem {
    uint32_t head[HSIZE];     // latest position (frame offset) per hash, NO_POS if none
    uint32_t ring[RING];      // bits not yet written out; ring[0] holds bit (flushed words * 32)
};

// One warp per segment g = b * nseg + s.  The chunk goes to slots + g * slot_bytes: length, "IDAT", data, CRC-32;
// seg_bytes[g] = its size.
__global__ void __launch_bounds__(32 * K9_WARPS) k9_png_deflate(const uint8_t* __restrict__ filt, int B, int H, int W,
                                                                uint8_t* __restrict__ slots, int64_t slot_bytes,
                                                                uint32_t* __restrict__ seg_bytes)
{
    extern __shared__ __align__(16) uint32_t k9_smem[];
    uint32_t* tab = k9_smem;                                               // CRC table, shared by the block
    for (int i = threadIdx.x; i < 256; i += blockDim.x) tab[i] = crc_table_entry(i);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nseg = segments(H);
    const int64_t g = (int64_t)blockIdx.x * K9_WARPS + warp;
    if (g >= (int64_t)B * nseg) return;
    DeflateSmem& sm = reinterpret_cast<DeflateSmem*>(k9_smem + 256)[warp];
    const int b = (int)(g / nseg), s = (int)(g % nseg);
    const int64_t stride = 1 + 2 * (int64_t)W;
    const uint8_t* f = filt + (int64_t)b * H * stride;
    int64_t s0, s1;
    segment_range(s, H, stride, &s0, &s1);
    const bool final_seg = s == nseg - 1;
    uint8_t* chunk = slots + g * slot_bytes;
    uint8_t* out = chunk + 8;
    uint32_t* outw = reinterpret_cast<uint32_t*>(out);
    const int64_t stored = stored_bytes(s1 - s0);

    for (int i = lane; i < HSIZE; i += 32) sm.head[i] = NO_POS;
    for (int i = lane; i < RING; i += 32) sm.ring[i] = i == 0 ? 2u : 0u;     // BFINAL 0, BTYPE 01
    __syncwarp();
    uint64_t bitpos = 3, flushed = 0;        // bits written, words moved out of the ring
    const int64_t hash_end = s1 - 2;         // positions with three bytes inside the segment
    int64_t chunk0 = s0, chunk_end = s0;     // positions hashed so far: [s0, chunk_end); cand holds [chunk0, chunk_end)
    uint32_t cand = NO_POS;                  // lane's: latest earlier position of the same hash, of position chunk0 + lane
    uint32_t tlen = 0, tval = 0;             // token number `lane` of the current batch
    int ntok = 0;
    bool aborted = false;

    // code the batch of ntok tokens into the ring, move the complete words out
    auto code_batch = [&](int n) {
        uint32_t bits = 0;
        const int nb = lane < n ? token_bits(tlen, tval, &bits) : 0;
        int incl = nb;
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        const int total = __shfl_sync(0xffffffffu, incl, 31);
        const uint64_t at = bitpos + (incl - nb);
        if (nb) {
            const int w = (int)((at >> 5) - flushed), sh = (int)(at & 31);
            atomicOr(&sm.ring[w], bits << sh);
            if (sh + nb > 32) atomicOr(&sm.ring[w + 1], bits >> (32 - sh));
        }
        __syncwarp();
        bitpos += total;
        const int full = (int)((bitpos >> 5) - flushed);
        if (lane < full) outw[flushed + lane] = sm.ring[lane];
        const uint32_t carry = sm.ring[full];
        __syncwarp();
        for (int i = lane; i < RING; i += 32) sm.ring[i] = i == 0 ? carry : 0u;
        __syncwarp();
        flushed += full;
    };

    int64_t p = s0;
    while (p < s1) {
        // hash every position below p + 1 (the table holds all earlier positions of the segment)
        while (p >= chunk_end) {
            chunk0 = chunk_end;
            const int64_t q = chunk0 + lane;
            const bool valid = q < hash_end;
            const unsigned vmask = __ballot_sync(0xffffffffu, valid);
            cand = NO_POS;
            uint32_t h = 0;
            unsigned peers = 0;
            if (valid) {
                h = hash3(f + q);
                peers = __match_any_sync(vmask, h);
                const unsigned before = peers & ((1u << lane) - 1);
                cand = before ? (uint32_t)(chunk0 + 31 - __clz(before)) : sm.head[h];
            }
            __syncwarp();
            if (valid && (peers >> lane) == 1u) sm.head[h] = (uint32_t)q;     // the group's latest position
            __syncwarp();
            chunk_end = chunk0 + 32;
        }
        const uint32_t qh = __shfl_sync(0xffffffffu, cand, (int)(p - chunk0));
        const int maxlen = (int)((s1 - p) < MAX_MATCH ? s1 - p : MAX_MATCH);
        int best_len = 0;
        int64_t best_d = 0;
        const uint8_t v0 = f[p];
        if (maxlen >= 3) {
            int64_t dist[4] = {1, 2, stride, qh != NO_POS ? p - (int64_t)qh : 0};
            unsigned alive = 0;
#pragma unroll
            for (int c = 0; c < 4; ++c)
                if (dist[c] > 0 && dist[c] <= p && dist[c] <= WINDOW) alive |= 1u << c;
            int lens[4] = {0, 0, 0, 0};
            for (int k = 0; alive && k < maxlen; k += 32) {
                const int i = k + lane;
                const bool in_range = i < maxlen;
                const uint8_t v = in_range ? f[p + i] : 0;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    if (!((alive >> c) & 1)) continue;
                    const bool eq = in_range && f[p - dist[c] + i] == v;
                    const unsigned miss = __ballot_sync(0xffffffffu, !eq);
                    if (miss) { lens[c] = k + __ffs(miss) - 1; alive &= ~(1u << c); }
                    else lens[c] = k + 32;
                }
            }
#pragma unroll
            for (int c = 0; c < 4; ++c)
                if (lens[c] >= 3 && (lens[c] > best_len || (lens[c] == best_len && dist[c] < best_d))) {
                    best_len = lens[c];
                    best_d = dist[c];
                }
        }
        if (lane == ntok) {
            tlen = (uint32_t)best_len;
            tval = best_len ? (uint32_t)best_d : v0;
        }
        p += best_len ? best_len : 1;
        if (++ntok == 32) {
            code_batch(32);
            ntok = 0;
            if ((int64_t)((bitpos + 10 + 7) >> 3) + 4 > stored) { aborted = true; break; }
        }
    }
    int64_t nbytes;
    if (!aborted) {
        if (ntok) code_batch(ntok);
        // end of block (7 zero bits), the empty stored block's header, byte alignment, LEN 0000 NLEN ffff
        bitpos += 7;
        const uint64_t hdr_at = bitpos;
        bitpos = ((bitpos + 3 + 7) >> 3) << 3;
        if (lane == 0) {
            const int w = (int)((hdr_at >> 5) - flushed), sh = (int)(hdr_at & 31);
            atomicOr(&sm.ring[w], (final_seg ? 1u : 0u) << sh);
            if (sh + 3 > 32) atomicOr(&sm.ring[w + 1], (final_seg ? 1u : 0u) >> (32 - sh));
            const int w2 = (int)((bitpos >> 5) - flushed), sh2 = (int)(bitpos & 31);
            atomicOr(&sm.ring[w2], 0xffff0000u << sh2);
            if (sh2) atomicOr(&sm.ring[w2 + 1], 0xffff0000u >> (32 - sh2));
        }
        __syncwarp();
        bitpos += 32;
        nbytes = (int64_t)(bitpos >> 3);
        const int words = (int)(((bitpos + 31) >> 5) - flushed);
        if (lane < words) outw[flushed + lane] = sm.ring[lane];
        __syncwarp();
        aborted = nbytes > stored;
    }
    if (aborted) {
        nbytes = write_stored(f, s0, s1, final_seg, out, lane, 32);
        __syncwarp();
    }
    // CRC-32 of "IDAT" + data: one piece per lane, combined pairwise across the lanes
    const int64_t per = (nbytes + 31) / 32;
    const int64_t a0 = lane * per < nbytes ? lane * per : nbytes;
    const int64_t a1 = a0 + per < nbytes ? a0 + per : nbytes;
    uint32_t crc = crc32_bytes(tab, 0, out + a0, a1 - a0);
    uint64_t len = (uint64_t)(a1 - a0);
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t c2 = __shfl_down_sync(0xffffffffu, crc, o);
        const uint64_t l2 = __shfl_down_sync(0xffffffffu, len, o);
        if ((lane & (2 * o - 1)) == 0 && lane + o < 32) {
            crc = crc32_combine(crc, c2, l2);
            len += l2;
        }
    }
    if (lane == 0) {
        const uint8_t idat[4] = {'I', 'D', 'A', 'T'};
        const uint32_t total_crc = crc32_combine(crc32_bytes(tab, 0, idat, 4), crc, (uint64_t)nbytes);
        put_be32(chunk, (uint32_t)nbytes);
        put_be32(chunk + 4, T_IDAT);
        put_be32(out + nbytes, total_crc);
        seg_bytes[g] = (uint32_t)(nbytes + 12);
    }
}

// One block: out_offsets[0..B] = exclusive scan of the file sizes (HEAD_BYTES + segment chunks + TAIL_BYTES)
__global__ void __launch_bounds__(1024) k9_png_offsets(const uint32_t* __restrict__ seg_bytes, int B, int nseg,
                                                       int64_t* __restrict__ out_offsets)
{
    __shared__ int64_t part[1024];
    const int t = threadIdx.x, n = blockDim.x;
    const int per = (B + n - 1) / n;
    const int b0 = t * per < B ? t * per : B, b1 = b0 + per < B ? b0 + per : B;
    int64_t sum = 0;
    for (int b = b0; b < b1; ++b) {
        sum += HEAD_BYTES + TAIL_BYTES;
        for (int s = 0; s < nseg; ++s) sum += seg_bytes[(int64_t)b * nseg + s];
    }
    part[t] = sum;
    __syncthreads();
    for (int o = 1; o < n; o <<= 1) {                 // inclusive scan of the threads' sums
        const int64_t v = t >= o ? part[t - o] : 0;
        __syncthreads();
        part[t] += v;
        __syncthreads();
    }
    int64_t off = part[t] - sum;
    for (int b = b0; b < b1; ++b) {
        out_offsets[b] = off;
        off += HEAD_BYTES + TAIL_BYTES;
        for (int s = 0; s < nseg; ++s) off += seg_bytes[(int64_t)b * nseg + s];
    }
    if (t == n - 1) out_offsets[B] = part[t];
}

// Block x = b * (nseg + 2) + j: j = 0 the header of file b, 1..nseg segment j-1's chunk, nseg+1 the Adler-32 and IEND
__global__ void __launch_bounds__(256) k9_png_pack(const uint8_t* __restrict__ slots, int64_t slot_bytes,
                                                   const uint32_t* __restrict__ seg_bytes,
                                                   const uint32_t* __restrict__ row_adler, int B, int H, int W,
                                                   const int64_t* __restrict__ out_offsets, uint8_t* __restrict__ out)
{
    __shared__ uint32_t tab[256];
    const int nseg = segments(H);
    const int64_t x = blockIdx.x;
    const int b = (int)(x / (nseg + 2)), j = (int)(x % (nseg + 2));
    if (b >= B) return;
    const uint32_t* sb = seg_bytes + (int64_t)b * nseg;
    uint8_t* o = out + out_offsets[b];
    if (j == 0 || j == nseg + 1) {
        for (int i = threadIdx.x; i < 256; i += blockDim.x) tab[i] = crc_table_entry(i);
        __syncthreads();
        if (threadIdx.x) return;
        if (j == 0) { write_head(o, tab, H, W); return; }
        const uint64_t stride = 1 + 2 * (uint64_t)W;
        uint32_t adler = 1;
        for (int r = 0; r < H; ++r) adler = adler32_combine(adler, row_adler[(int64_t)b * H + r], stride);
        int64_t pos = HEAD_BYTES;
        for (int s = 0; s < nseg; ++s) pos += sb[s];
        write_tail(o + pos, tab, adler);
        return;
    }
    const int s = j - 1;
    int64_t pos = HEAD_BYTES;
    for (int k = 0; k < s; ++k) pos += sb[k];
    const uint8_t* src = slots + ((int64_t)b * nseg + s) * slot_bytes;
    const uint32_t n = sb[s];
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) o[pos + i] = src[i];
}

}  // namespace png
}  // namespace dtfill
