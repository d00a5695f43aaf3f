// dtfill_k8_png.cuh -- batched decoder of 16-bit grayscale PNG files (KITTI depth maps, data_read.py:215 reads them
// with PIL), so that a batch of compressed files becomes uint16 samples [B,H,W] on the device.
//
// Supported input, and nothing more: colour type 0, bit depth 16, compression 0, filter method 0, no interlace; any
// mix of the five row filters; any DEFLATE content (stored, fixed and dynamic Huffman blocks); the zlib stream split
// over any number of IDAT chunks (empty ones included); ancillary chunks anywhere before IEND are skipped.  Chunk
// CRC-32s are NOT checked: the Adler-32 of the zlib stream covers the image data.
//
//   k8_png_inflate   one warp per file.  Lane 0 walks the chunks, checks the IHDR against the batch's (H, W) and the
//                    zlib header, and decodes Huffman symbols serially into a shared queue of tokens (literal runs,
//                    matches); the whole warp then expands the queue into the frame's scratch of H*(1+2W) filtered
//                    bytes, one token after the other (a match may read what the token before it wrote), a match as
//                    dst[p+i] = dst[p-d+(i mod d)] so that all lanes copy at once even when d < len (runs of zero
//                    bytes at distance 1-2 are the common case here).  The Adler-32 is summed by the lanes from the
//                    bytes they store.
//   k8_png_unfilter  one warp per frame, a 32-row wavefront: lane k owns row r0+k and runs one sample behind lane
//                    k-1, from which it takes the row above by shuffles, so None/Sub/Up/Average/Paeth rows all take
//                    the same path.  Samples are swapped from PNG's big-endian order to native uint16.
//
// Bounds: every decision that could take a read outside the file or a write outside the frame is made by the serial
// token decoder before the token is queued (over-subscribed / incomplete code sets, symbols 286-287 and distance codes
// 30-31, a distance before the start of the output, output beyond H*(1+2W), LEN != ~NLEN, running out of input).  The
// bit reader, the Huffman tables and the token decoder are __host__ __device__: dtfill_debug_png_decode_host runs the
// same code serially on the CPU.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace dtfill {
namespace png {

// per-frame status codes (include/dtfill.h dtfill_png_decode)
enum : int {
    ST_OK = 0, ST_SIGNATURE = 1, ST_IHDR = 2, ST_SIZE = 3, ST_CHUNKS = 4, ST_ZLIB = 5, ST_DEFLATE = 6, ST_LENGTH = 7,
    ST_FILTER = 8, ST_ADLER = 9
};

constexpr int LBITS = 10;            // primary lookup bits of the literal/length table
constexpr int DBITS = 9;             // ... of the distance (and code-length) table
constexpr int QCAP = 64;             // tokens per round of the warp
constexpr int LITCAP = 256;          // literal bytes per round
constexpr uint32_t LIT_RUN = 0x80000000u;   // token arg flag: a run of literals at lit[arg & 0xffff]
constexpr uint32_t ADLER_MOD = 65521u;

#define PNG_HD __host__ __device__ __forceinline__

PNG_HD uint32_t be32(const uint8_t* p) {
    return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | (uint32_t)p[3];
}

constexpr uint32_t T_IHDR = 0x49484452u, T_IDAT = 0x49444154u, T_IEND = 0x49454e44u;

// Signature, IHDR, chunk structure of one file of n bytes.  On success *first_idat is the offset of the first IDAT
// chunk's length field.  A file whose IHDR is valid but whose size differs from (H, W) is ST_SIZE.
PNG_HD int check_structure(const uint8_t* f, int64_t n, int H, int W, int64_t* first_idat) {
    const uint8_t sig[8] = {137, 80, 78, 71, 13, 10, 26, 10};
    if (n < 8) return ST_SIGNATURE;
    for (int i = 0; i < 8; ++i)
        if (f[i] != sig[i]) return ST_SIGNATURE;
    if (n < 8 + 8 + 13 + 4 || be32(f + 8) != 13 || be32(f + 12) != T_IHDR) return ST_CHUNKS;
    const uint8_t* ih = f + 16;
    if (ih[8] != 16 || ih[9] != 0 || ih[10] != 0 || ih[11] != 0 || ih[12] != 0) return ST_IHDR;
    const uint32_t w = be32(ih), hh = be32(ih + 4);
    if (w == 0 || hh == 0 || w > 0x7fffffffu || hh > 0x7fffffffu) return ST_IHDR;
    int size_st = (w != (uint32_t)W || hh != (uint32_t)H) ? ST_SIZE : ST_OK;
    int64_t pos = 33, idat = -1;
    for (;;) {
        if (pos + 12 > n) return ST_CHUNKS;                       // length, type, CRC
        const uint32_t len = be32(f + pos), type = be32(f + pos + 4);
        if (len > 0x7fffffffu || (int64_t)len > n - pos - 12) return ST_CHUNKS;
        if (type == T_IEND) break;
        if (type == T_IHDR) return ST_CHUNKS;
        if (type == T_IDAT) { if (idat < 0) idat = pos; }
        else if (!(f[pos + 4] & 0x20)) return ST_CHUNKS;           // unknown critical chunk (PLTE has no place here)
        pos += 12 + (int64_t)len;
    }
    if (idat < 0) return ST_CHUNKS;
    *first_idat = idat;
    return size_st;
}

// Bytes of the concatenated IDAT payloads, read across chunk boundaries (the structure was checked before).
struct IdatReader {
    const uint8_t* f;
    int64_t pos, end;        // current payload byte, end of the current payload (its CRC)
    bool eof;
};

PNG_HD void idat_open(IdatReader& r, const uint8_t* f, int64_t first_idat) {
    r.f = f; r.pos = r.end = first_idat - 4; r.eof = false;
}

PNG_HD int idat_byte(IdatReader& r) {
    while (r.pos == r.end) {
        if (r.eof) return -1;
        const int64_t c = r.end + 4;                  // next chunk's length field
        const uint32_t len = be32(r.f + c), type = be32(r.f + c + 4);
        if (type == T_IEND) { r.eof = true; return -1; }
        r.end = c + 8 + len;
        r.pos = (type == T_IDAT) ? c + 8 : r.end;
    }
    return r.f[r.pos++];
}

// LSB-first bit reader over the IDAT bytes.  Past the end it shifts in zeros and counts them in `over`: the stream ran
// out of input as soon as more bits were consumed than were real (over > cnt).
struct Bits {
    IdatReader in;
    uint64_t buf;
    int cnt;
    int over;
};

PNG_HD void refill(Bits& b) {
    while (b.cnt <= 56) {
        int c = idat_byte(b.in);
        if (c < 0) { c = 0; b.over += 8; }
        b.buf |= (uint64_t)c << b.cnt;
        b.cnt += 8;
    }
}
PNG_HD bool overrun(const Bits& b) { return b.over > b.cnt; }
PNG_HD uint32_t peek(const Bits& b, int n) { return (uint32_t)(b.buf & ((1ull << n) - 1)); }
PNG_HD void drop(Bits& b, int n) { b.buf >>= n; b.cnt -= n; }
PNG_HD uint32_t take(Bits& b, int n) { uint32_t v = peek(b, n); drop(b, n); return v; }

// Canonical Huffman code: primary table of 2^tbits entries (symbol << 4 | length, 0 for codes longer than tbits),
// counts per length and symbols sorted by (length, value) for the longer codes.
struct Huff {
    uint16_t* lut;
    uint16_t* count;     // [16]
    uint16_t* sym;
    int tbits;
};

// kind 0: code-length code (must be complete); 1: literal/length or distance code (zlib's rule: a single code of
// length 1 may stand alone, and a code without symbols is accepted until it is used).  Returns false when the
// lengths are over-subscribed or incomplete.
PNG_HD bool build_huff(Huff& h, const uint8_t* lens, int n, int kind) {
    for (int l = 0; l < 16; ++l) h.count[l] = 0;
    for (int s = 0; s < n; ++s) h.count[lens[s]]++;
    h.count[0] = 0;
    int left = 1, maxl = 0;
    for (int l = 1; l < 16; ++l) {
        left <<= 1;
        left -= h.count[l];
        if (left < 0) return false;                 // over-subscribed
        if (h.count[l]) maxl = l;
    }
    if (left > 0 && (kind == 0 || maxl != 1) && maxl != 0) return false;   // incomplete
    if (maxl == 0 && kind == 0) return false;
    uint16_t offs[16];
    offs[1] = 0;
    for (int l = 1; l < 15; ++l) offs[l + 1] = offs[l] + h.count[l];
    for (int s = 0; s < n; ++s)
        if (lens[s]) h.sym[offs[lens[s]]++] = (uint16_t)s;
    const int size = 1 << h.tbits;
    for (int i = 0; i < size; ++i) h.lut[i] = 0;
    // canonical codes in (length, symbol) order; the table is indexed by the bit-reversed code
    int code = 0, idx = 0;
    for (int l = 1; l <= h.tbits; ++l) {
        for (int k = 0; k < h.count[l]; ++k, ++idx, ++code) {
            int rev = 0;
            for (int j = 0; j < l; ++j) rev |= ((code >> j) & 1) << (l - 1 - j);
            const uint16_t e = (uint16_t)((h.sym[idx] << 4) | l);
            for (int i = rev; i < size; i += 1 << l) h.lut[i] = e;
        }
        code <<= 1;
    }
    return true;
}

// Next symbol (the buffer holds at least 15 bits); -1: no code matches.
PNG_HD int decode_sym(Bits& b, const Huff& h) {
    const uint32_t e = h.lut[peek(b, h.tbits)];
    if (e & 15) { drop(b, e & 15); return (int)(e >> 4); }
    int code = 0, first = 0, index = 0;
    for (int l = 1; l < 16; ++l) {
        code |= (int)((b.buf >> (l - 1)) & 1);
        const int c = h.count[l];
        if (code - c < first) { drop(b, l); return h.sym[index + (code - first)]; }
        index += c; first += c; first <<= 1; code <<= 1;
    }
    return -1;
}

// Token queue of one round: len[i] bytes; arg[i] = match distance, or LIT_RUN | offset into lit.
struct Queue {
    uint32_t* len;
    uint32_t* arg;
    uint8_t* lit;
    int n, nlit;
};

struct Inflate {
    Bits b;
    uint32_t out, total;     // bytes queued so far, bytes the frame must have
    int state;               // 0: block header next, 1: Huffman block, 2: stored block, 3: after the final block
    int final_blk;
    uint32_t stored_left;
    uint32_t adler;          // the trailer, once state == 3
};

PNG_HD void queue_literal(Queue& q, uint8_t v) {
    if (q.n > 0 && (q.arg[q.n - 1] & LIT_RUN) && (q.arg[q.n - 1] & 0xffff) + q.len[q.n - 1] == (uint32_t)q.nlit) {
        q.len[q.n - 1]++;
    } else {
        q.len[q.n] = 1;
        q.arg[q.n] = LIT_RUN | (uint32_t)q.nlit;
        q.n++;
    }
    q.lit[q.nlit++] = v;
}

PNG_HD void fixed_tables(Huff& lh, Huff& dh, uint8_t* lens) {
    for (int i = 0; i < 144; ++i) lens[i] = 8;
    for (int i = 144; i < 256; ++i) lens[i] = 9;
    for (int i = 256; i < 280; ++i) lens[i] = 7;
    for (int i = 280; i < 288; ++i) lens[i] = 8;
    build_huff(lh, lens, 288, 1);
    for (int i = 0; i < 32; ++i) lens[i] = 5;
    build_huff(dh, lens, 32, 1);
}

// Dynamic block header: code-length code, then the literal/length and distance code lengths.
PNG_HD int dynamic_tables(Bits& b, Huff& lh, Huff& dh, uint8_t* lens) {
    static constexpr uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    refill(b);
    const int nlen = (int)take(b, 5) + 257, ndist = (int)take(b, 5) + 1, ncode = (int)take(b, 4) + 4;
    if (nlen > 286 || ndist > 30) return ST_DEFLATE;
    for (int i = 0; i < 19; ++i) lens[i] = 0;
    for (int i = 0; i < ncode; ++i) {
        refill(b);
        lens[order[i]] = (uint8_t)take(b, 3);
    }
    if (overrun(b)) return ST_DEFLATE;
    if (!build_huff(dh, lens, 19, 0)) return ST_DEFLATE;     // the distance table holds the code-length code for now
    uint8_t* all = lens + 19;                                 // nlen + ndist lengths
    int i = 0;
    while (i < nlen + ndist) {
        refill(b);
        const int s = decode_sym(b, dh);
        if (s < 0) return ST_DEFLATE;
        if (s < 16) { all[i++] = (uint8_t)s; continue; }
        int rep, v = 0;
        if (s == 16) {
            if (i == 0) return ST_DEFLATE;
            v = all[i - 1];
            rep = 3 + (int)take(b, 2);
        } else if (s == 17) {
            rep = 3 + (int)take(b, 3);
        } else {
            rep = 11 + (int)take(b, 7);
        }
        if (i + rep > nlen + ndist) return ST_DEFLATE;
        while (rep--) all[i++] = (uint8_t)v;
    }
    if (overrun(b)) return ST_DEFLATE;
    if (all[256] == 0) return ST_DEFLATE;                     // no end-of-block code
    if (!build_huff(lh, all, nlen, 1)) return ST_DEFLATE;
    if (!build_huff(dh, all + nlen, ndist, 1)) return ST_DEFLATE;
    return ST_OK;
}

// zlib header: CM 8, CINFO <= 7, FCHECK, no preset dictionary.
PNG_HD int zlib_header(Inflate& s) {
    refill(s.b);
    const uint32_t cmf = take(s.b, 8), flg = take(s.b, 8);
    if (overrun(s.b)) return ST_ZLIB;
    if ((cmf & 15) != 8 || (cmf >> 4) > 7 || ((cmf << 8) | flg) % 31 != 0 || (flg & 0x20)) return ST_ZLIB;
    return ST_OK;
}

// Decode tokens into q until it is full or the stream ends (state 3).  Returns a status; nothing it queued lies
// outside [0, total) or reads before the start of the output.
PNG_HD int inflate_tokens(Inflate& s, Huff& lh, Huff& dh, uint8_t* lens, Queue& q) {
    static constexpr uint16_t lbase[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59,
                                           67, 83, 99, 115, 131, 163, 195, 227, 258};
    static constexpr uint8_t lext[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
    static constexpr uint16_t dbase[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769,
                                           1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
    static constexpr uint8_t dext[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11,
                                         11, 12, 12, 13, 13};
    q.n = 0;
    q.nlit = 0;
    while (q.n < QCAP && q.nlit < LITCAP) {
        if (s.state == 3) return ST_OK;
        if (s.state == 0) {
            refill(s.b);
            s.final_blk = (int)take(s.b, 1);
            const int type = (int)take(s.b, 2);
            if (type == 0) {
                drop(s.b, s.b.cnt & 7);                       // to the byte boundary
                refill(s.b);
                const uint32_t len = take(s.b, 16), nlen = take(s.b, 16);
                if (overrun(s.b)) return ST_DEFLATE;
                if (len != (~nlen & 0xffffu)) return ST_DEFLATE;
                s.stored_left = len;
                s.state = 2;
            } else if (type == 1) {
                fixed_tables(lh, dh, lens);
                s.state = 1;
            } else if (type == 2) {
                const int st = dynamic_tables(s.b, lh, dh, lens);
                if (st) return st;
                s.state = 1;
            } else {
                return ST_DEFLATE;
            }
            if (overrun(s.b)) return ST_DEFLATE;
        }
        if (s.state == 2) {
            while (s.stored_left && q.n < QCAP && q.nlit < LITCAP) {
                if (s.out >= s.total) return ST_LENGTH;
                refill(s.b);
                const uint8_t v = (uint8_t)take(s.b, 8);
                if (overrun(s.b)) return ST_DEFLATE;
                queue_literal(q, v);
                s.out++;
                s.stored_left--;
            }
            if (s.stored_left == 0) s.state = s.final_blk ? 3 : 0;
            continue;
        }
        // Huffman block: one literal or one match per iteration (at most 48 bits, one refill)
        refill(s.b);
        const int sym = decode_sym(s.b, lh);
        if (sym < 0) return ST_DEFLATE;
        if (sym < 256) {
            if (s.out >= s.total) return ST_LENGTH;
            queue_literal(q, (uint8_t)sym);
            s.out++;
        } else if (sym == 256) {
            s.state = s.final_blk ? 3 : 0;
        } else {
            if (sym > 285) return ST_DEFLATE;
            const int li = sym - 257;
            const uint32_t len = lbase[li] + take(s.b, lext[li]);
            const int ds = decode_sym(s.b, dh);
            if (ds < 0 || ds > 29) return ST_DEFLATE;
            const uint32_t dist = dbase[ds] + take(s.b, dext[ds]);
            if (overrun(s.b)) return ST_DEFLATE;
            if (dist > s.out) return ST_DEFLATE;              // before the start of the output
            if (len > s.total - s.out) return ST_LENGTH;
            q.len[q.n] = len;
            q.arg[q.n] = dist;
            q.n++;
            s.out += len;
        }
        if (overrun(s.b)) return ST_DEFLATE;
    }
    return ST_OK;
}

// After the final block: the output must be complete, then the Adler-32 trailer (big-endian, byte aligned).
PNG_HD int finish(Inflate& s) {
    if (s.out != s.total) return ST_LENGTH;
    drop(s.b, s.b.cnt & 7);
    refill(s.b);
    uint32_t a = 0;
    for (int i = 0; i < 4; ++i) a = (a << 8) | take(s.b, 8);
    if (overrun(s.b)) return ST_DEFLATE;
    s.adler = a;
    return ST_OK;
}

PNG_HD int paeth(int a, int b, int c) {
    const int p = a + b - c;
    const int pa = p > a ? p - a : a - p, pb = p > b ? p - b : b - p, pc = p > c ? p - c : c - p;
    return (pa <= pb && pa <= pc) ? a : (pb <= pc ? b : c);
}

// One byte of a row: x filtered, a left, b above, c above-left (bytes of the same significance)
PNG_HD uint32_t unfilter_byte(int ft, uint32_t x, uint32_t a, uint32_t b, uint32_t c) {
    switch (ft) {
        case 1: return (x + a) & 255;
        case 2: return (x + b) & 255;
        case 3: return (x + ((a + b) >> 1)) & 255;
        case 4: return (x + (uint32_t)paeth((int)a, (int)b, (int)c)) & 255;
        default: return x;
    }
}

// One 16-bit sample from its two filtered bytes and the three neighbouring samples.
PNG_HD uint32_t unfilter_sample(int ft, uint32_t xh, uint32_t xl, uint32_t a, uint32_t b, uint32_t c) {
    const uint32_t hi = unfilter_byte(ft, xh, a >> 8, b >> 8, c >> 8);
    const uint32_t lo = unfilter_byte(ft, xl, a & 255, b & 255, c & 255);
    return (hi << 8) | lo;
}

struct __align__(16) InflateSmem {
    uint16_t llut[1 << LBITS];
    uint16_t dlut[1 << DBITS];
    uint16_t lsym[288];
    uint16_t dsym[32];
    uint16_t lcount[16];
    uint16_t dcount[16];
    uint32_t qlen[QCAP];
    uint32_t qarg[QCAP];
    uint8_t lens[19 + 320];
    uint8_t lit[LITCAP];
};

constexpr int K8_WARPS = 4;

// One warp per file b of data[offsets[b], offsets[b+1]): filtered bytes [H*(1+2W)] into scr + b*H*(1+2W), status[b].
__global__ void __launch_bounds__(32 * K8_WARPS) k8_png_inflate(const uint8_t* __restrict__ data,
                                                                const int64_t* __restrict__ offsets, int B, int H, int W,
                                                                uint8_t* scr, int32_t* __restrict__ status)
{
    __shared__ InflateSmem sm_all[K8_WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * K8_WARPS + warp;
    if (b >= B) return;
    InflateSmem& sm = sm_all[warp];
    const uint32_t total = (uint32_t)H * (uint32_t)(1 + 2 * W);
    uint8_t* dst = scr + (size_t)b * total;

    Inflate s;
    Huff lh{sm.llut, sm.lcount, sm.lsym, LBITS}, dh{sm.dlut, sm.dcount, sm.dsym, DBITS};
    Queue q{sm.qlen, sm.qarg, sm.lit, 0, 0};
    int st = ST_OK;
    if (lane == 0) {
        const int64_t o0 = offsets[b], o1 = offsets[b + 1];
        int64_t first = 0;
        st = o1 < o0 ? ST_CHUNKS : check_structure(data + o0, o1 - o0, H, W, &first);
        if (st == ST_OK) {
            s.b.buf = 0; s.b.cnt = 0; s.b.over = 0;
            idat_open(s.b.in, data + o0, first);
            s.out = 0; s.total = total; s.state = 0; s.final_blk = 0; s.stored_left = 0; s.adler = 0;
            st = zlib_header(s);
        }
    }
    st = __shfl_sync(0xffffffffu, st, 0);
    uint64_t sa = 0, sb = 0;      // this lane's share of the Adler-32 sums: sum of x_p, sum of (total - p) * x_p
    uint32_t p = 0;
    bool done = st != ST_OK;
    while (!done) {
        int n = 0, state = 0;
        if (lane == 0) {
            st = inflate_tokens(s, lh, dh, sm.lens, q);
            n = q.n;
            state = s.state;
        }
        __syncwarp();
        st = __shfl_sync(0xffffffffu, st, 0);
        n = __shfl_sync(0xffffffffu, n, 0);
        state = __shfl_sync(0xffffffffu, state, 0);
        for (int i = 0; i < n; ++i) {
            const uint32_t len = sm.qlen[i], arg = sm.qarg[i];
            if (arg & LIT_RUN) {
                const uint8_t* lit = sm.lit + (arg & 0xffff);
                for (uint32_t j = lane; j < len; j += 32) {
                    const uint32_t v = lit[j];
                    dst[p + j] = (uint8_t)v;
                    sa += v;
                    sb += (uint64_t)(total - p - j) * v;
                }
            } else {
                const uint32_t d = arg;
                for (uint32_t j = lane; j < len; j += 32) {
                    const uint32_t v = dst[p - d + (j < d ? j : j % d)];
                    dst[p + j] = (uint8_t)v;
                    sa += v;
                    sb += (uint64_t)(total - p - j) * v;
                }
            }
            p += len;
            __syncwarp();      // the next token may read these bytes
        }
        done = st != ST_OK || state == 3;
    }
    if (st == ST_OK && lane == 0) st = finish(s);
    st = __shfl_sync(0xffffffffu, st, 0);
    if (st == ST_OK) {
        uint32_t a32 = (uint32_t)(sa % ADLER_MOD), b32 = (uint32_t)(sb % ADLER_MOD);
        for (int o = 16; o; o >>= 1) {
            a32 += __shfl_xor_sync(0xffffffffu, a32, o);
            b32 += __shfl_xor_sync(0xffffffffu, b32, o);
        }
        if (lane == 0) {
            const uint32_t A = (1u + a32) % ADLER_MOD, Bv = (uint32_t)(((uint64_t)total + b32) % ADLER_MOD);
            if (((Bv << 16) | A) != s.adler) st = ST_ADLER;
        }
    }
    if (lane == 0) status[b] = st;
}

// One warp per frame: filtered bytes -> native uint16 samples [H,W]; frames whose status is not 0 are zeroed.
__global__ void __launch_bounds__(32 * K8_WARPS) k8_png_unfilter(const uint8_t* __restrict__ scr, int B, int H, int W,
                                                                 uint16_t* __restrict__ out, int32_t* __restrict__ status)
{
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * K8_WARPS + warp;
    if (b >= B) return;
    const size_t stride = (size_t)(1 + 2 * W);
    const uint8_t* f = scr + (size_t)b * H * stride;
    uint16_t* o = out + (size_t)b * H * W;
    int st = status[b];
    if (st == ST_OK) {
        bool bad = false;
        for (int r = lane; r < H; r += 32) bad |= f[r * stride] > 4;
        if (__any_sync(0xffffffffu, bad)) {
            st = ST_FILTER;
            if (lane == 0) status[b] = st;
        }
    }
    if (st != ST_OK) {
        for (size_t i = lane; i < (size_t)H * W; i += 32) o[i] = 0;
        return;
    }
    for (int r0 = 0; r0 < H; r0 += 32) {
        const int r = r0 + lane;
        const bool active = r < H;
        const uint8_t* row = f + (size_t)(active ? r : 0) * stride;
        const int ft = active ? row[0] : 0;
        ++row;
        const uint16_t* above = o + (size_t)(r0 > 0 ? r0 - 1 : 0) * W;      // read through upv when r0 > 0
        uint32_t cur = 0, prev = 0;            // this lane's last two reconstructed samples (columns c-1, c-2)
        uint32_t upv = 0, upnext = 0, uplast = 0;
        if (r0 > 0 && lane < W) upnext = above[lane];
        for (int t = 0; t < W + 31; ++t) {
            if ((t & 31) == 0) {                  // lane 0's row above, 32 columns at a time, one chunk ahead
                uplast = __shfl_sync(0xffffffffu, upv, 31);
                upv = upnext;
                const int c2 = t + 32 + lane;
                upnext = (r0 > 0 && c2 < W) ? above[c2] : 0;
            }
            const uint32_t up_k = __shfl_up_sync(0xffffffffu, cur, 1);
            const uint32_t ul_k = __shfl_up_sync(0xffffffffu, prev, 1);
            const uint32_t up_0 = __shfl_sync(0xffffffffu, upv, t & 31);
            const uint32_t ul_0 = __shfl_sync(0xffffffffu, upv, (t - 1) & 31);
            const int c = t - lane;
            if (active && c >= 0 && c < W) {
                const uint32_t up = lane ? up_k : up_0;
                const uint32_t ul = lane ? ul_k : (c == 0 ? 0u : ((t & 31) ? ul_0 : uplast));
                const uint32_t v = unfilter_sample(ft, row[2 * c], row[2 * c + 1], cur, up, ul);
                o[(size_t)r * W + c] = (uint16_t)v;
                prev = cur;
                cur = v;
            }
        }
        __syncwarp();
    }
}

}  // namespace png
}  // namespace dtfill
