// dtfill_k1b_plan.cuh -- K1b: per-frame scans, depth_list (tools.py:24), tile planner
#pragma once
#include "dtfill_common.cuh"

namespace dtfill {

// ------------------------------------------------------------------------------------------------------
// K1b: per frame -- exclusive scans of the row counts, depth_list compaction, task emission.
// One 256-thread block per frame.
// ------------------------------------------------------------------------------------------------------
constexpr int K1B_THREADS = 512;

__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* smem /*[K1B_THREADS/32 + 1]*/, uint32_t& total)
{
    constexpr int NW = K1B_THREADS / 32;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += o;
    }
    if (lane == 31) smem[wid] = inc;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t run = 0;
        for (int i = 0; i < NW; ++i) { const uint32_t t = smem[i]; smem[i] = run; run += t; }
        smem[NW] = run;
    }
    __syncthreads();
    const uint32_t base = smem[wid];
    total = smem[NW];
    __syncthreads();
    return base + inc - v;
}

// barrier among the 256 planner threads only (warps 8..15), so that the compaction warps are not held up
__device__ __forceinline__ void planner_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

__global__ void __launch_bounds__(K1B_THREADS) k1b_scan_compact(FrameParams fp, Workspace ws,
                                                                 int32_t* __restrict__ out_counts)
{
    __shared__ uint32_t sm[K1B_THREADS / 32 + 1];
    __shared__ uint16_t cellD[MAX_CELLS];        // planner: distance (pixels) to the nearest occupied cell
    __shared__ int cellU[1024];                  // planner: per cell-row upper bound of dt
    __shared__ uint32_t srcrows[128];            // planner: bit y = row y holds a source (H <= 4096)
    __shared__ Task st[MAXT];                    // planner: tasks of this frame before ordering
    __shared__ int scost[MAXT];
    __shared__ int snt;
    DTFILL_TRACE_SCOPE(fp, 1);
    const int b = blockIdx.x;
    const int H = fp.H, W = fp.W, WW = fp.WW;
    const int tid = threadIdx.x;
    const int lane = tid & 31, wid = tid >> 5;
    const int per = (H + K1B_THREADS - 1) / K1B_THREADS;
    const int y0 = min(H, tid * per), y1 = min(H, y0 + per);
    uint32_t* rs = ws.rowsrc + (long)b * H;
    uint32_t* rv = ws.rowval + (long)b * H;

#ifdef DTFILL_PLANNER_CLOCKS     // phase clocks of block 0 (profiles/k1b_clock.py reads them through dtfill_debug_read_status)
    const long long dbg_t0 = clock64();
    auto dbg_mark = [&](int k) { if (b == 0 && (tid == 0 || tid == 256)) ws.status[4 + k + (tid ? 8 : 0)] = (int)(clock64() - dbg_t0); };
#else
    auto dbg_mark = [](int) {};
#endif
    if (tid < 128) srcrows[tid] = 0;
    uint32_t ls = 0, lv = 0;
    for (int y = y0; y < y1; ++y) { ls += rs[y]; lv += rv[y]; }
    uint32_t nsrc, nval;
    uint32_t bs = block_exclusive_scan(ls, sm, nsrc);
    uint32_t bv = block_exclusive_scan(lv, sm, nval);
    for (int y = y0; y < y1; ++y) {
        const uint32_t s_ = rs[y], v_ = rv[y];
        rs[y] = bs; rv[y] = bv;
        bs += s_; bv += v_;
        if (s_ && y < 4096) atomicOr(&srcrows[y >> 5], 1u << (y & 31));
    }
    __syncthreads();

    dbg_mark(0);
    const int B = fp.B;
    int kind = (nsrc == 0) ? TASK_NOSRC : ((fp.force_wide || nsrc > MAX_FAST_LABEL) ? TASK_WIDE : TASK_CHAMFER);
    if (nval == 0) kind = TASK_SKIP;
    const int nh = (H + CELL_H - 1) / CELL_H, nw = (W + CELL_W - 1) / CELL_W;
    const bool plan = kind == TASK_CHAMFER && fp.band_cap > 0 && nh * nw <= MAX_CELLS && nh <= 1024 && H <= 4096 &&
                      2 * H > fp.band_cap;

    // Rows above the first source row f need no scan (k3_sky): S0 = rows handed over, a multiple of the cell height
    // with S0 + 1 <= f.  The planner's grid then starts at cell row c0row: cells above hold no source and lie on no
    // shortest path between a cell and a source below them.
    int S0 = 0;
    if (plan && fp.sky_min > 0 && W <= SKY_MAX_W) {
        int f = 0;
        for (int w = 0; w < 128 && (w << 5) < H; ++w)
            if (srcrows[w]) { f = (w << 5) + __ffs(srcrows[w]) - 1; break; }
        const int s4 = f >= 1 ? ((f - 1) / CELL_H) * CELL_H : 0;
        if (s4 >= fp.sky_min) S0 = s4;
    }
    const int c0row = S0 / CELL_H;

    if (wid < 8) {
        // ---- warps 0..7: depth_list = in[valid] in raster order (tools.py:24).  K1 left every row's valid depths
        // compacted at the start of the row's slot in ws.scratch; concatenate the non-empty rows.
        float* dl = ws.dlist + (long)b * H * W;
        const float* rowvals = reinterpret_cast<const float*>(ws.scratch) + (long)b * H * W;
        for (int yb = wid * 32; yb < H; yb += 8 * 32) {
            // one coalesced read of 33 row bases per 32 rows instead of two dependent loads per row
            const int yy = yb + lane;
            const uint32_t mybase = yy < H ? rv[yy] : nval;
            const uint32_t nextbase = __shfl_down_sync(0xffffffffu, mybase, 1);
            const uint32_t after = (yb + 32 < H) ? rv[yb + 32] : nval;
            const uint32_t mycnt = (lane == 31 ? after : nextbase) - mybase;
            for (int r = 0; r < 32 && yb + r < H; ++r) {
                const uint32_t cnt = __shfl_sync(0xffffffffu, mycnt, r);
                if (cnt == 0) continue;
                const uint32_t base = __shfl_sync(0xffffffffu, mybase, r);
                const float* src = rowvals + (long)(yb + r) * W + lane;
                float* dst = dl + base + lane;
                for (uint32_t i0 = 0; i0 < cnt; i0 += 32 * 12) {       // 12 loads in flight per lane
                    const int rem = (int)(cnt - i0) - lane;            // elements k with 32 k < rem are this lane's
                    const float* sp = src + i0;
                    float* dp = dst + i0;
                    float v[12];
#pragma unroll
                    for (int k = 0; k < 12; ++k) v[k] = 32 * k < rem ? sp[32 * k] : 0.f;
#pragma unroll
                    for (int k = 0; k < 12; ++k)
                        if (32 * k < rem) dp[32 * k] = v[k];
                }
            }
        }
        dbg_mark(1);
        return;
    }

    // ---- warps 8..15: tile planner -------------------------------------------------------------------------
    const int ptid = tid - 256, pw = wid - 8;
    if (plan) {
        // coarse occupancy -> exact anisotropic city-block distance on the cell grid (two sweeps per axis)
        // rowcell nibbles of CELL_H consecutive rows OR-ed per word, then one distance cell per bit
        const uint8_t* rc = ws.rowcell + (long)b * H * WW;
        // one warp per cell row, two cell rows per turn, a lane per word: the CELL_H rows' nibbles OR-ed and expanded
        // into the word's four distance cells at once (no index division, 8 byte loads in flight per lane)
        for (int cy0 = c0row + pw; cy0 < nh; cy0 += 16) {
            for (int w0 = 0; w0 < WW; w0 += 32) {
                const int w = w0 + lane;
                uint32_t o[2] = {0u, 0u};
#pragma unroll
                for (int t = 0; t < 2; ++t) {
                    const int cy = cy0 + 8 * t;
#pragma unroll
                    for (int r = 0; r < CELL_H; ++r) {
                        const int y = cy * CELL_H + r;
                        if (cy < nh && y < H && w < WW) o[t] |= rc[(long)y * WW + w];
                    }
                }
#pragma unroll
                for (int t = 0; t < 2; ++t) {
                    const int cy = cy0 + 8 * t;
                    if (cy < nh && w < WW) {
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            if (4 * w + j < nw) cellD[cy * nw + 4 * w + j] = ((o[t] >> j) & 1u) ? 0 : 60000;
                    }
                }
            }
        }
        planner_sync();
        dbg_mark(2);
        for (int cx = ptid; cx < nw; cx += 256) {        // vertical sweeps, one thread per cell column
            uint32_t d = 60000;
            for (int c0 = c0row; c0 < nh; c0 += 8) {     // 8 loads ahead of the dependent (min,+) chain
                uint32_t v[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) v[k] = c0 + k < nh ? (uint32_t)cellD[(c0 + k) * nw + cx] : 60000u;
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    d = min(min(d + CELL_H, v[k]), 60000u);
                    if (c0 + k < nh) cellD[(c0 + k) * nw + cx] = (uint16_t)d;
                }
            }
            d = 60000;
            for (int c0 = nh - 1; c0 >= c0row; c0 -= 8) {
                uint32_t v[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) v[k] = c0 - k >= c0row ? (uint32_t)cellD[(c0 - k) * nw + cx] : 60000u;
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    d = min(min(d + CELL_H, v[k]), 60000u);
                    if (c0 - k >= c0row) cellD[(c0 - k) * nw + cx] = (uint16_t)d;
                }
            }
        }
        planner_sync();
        dbg_mark(3);
        // horizontal sweeps, one warp per cell row: a lane keeps its (up to 8) consecutive cells in registers,
        // (min,+) scans across lanes via shuffles; only the row maximum leaves the warp
        const int chunk = (nw + 31) / 32;
        if (chunk <= 8) {
            // two cell rows per warp and turn, their (independent) chains interleaved
            for (int cy0 = c0row + pw; cy0 < nh; cy0 += 16) {
                const int xa = lane * chunk;
                uint32_t v[2][8], d[2], e[2], mx[2];
#pragma unroll
                for (int t = 0; t < 2; ++t) {
                    const int cy = cy0 + 8 * t;
                    const uint16_t* rowp = cellD + (cy < nh ? cy : cy0) * nw;
#pragma unroll
                    for (int k = 0; k < 8; ++k) v[t][k] = (k < chunk && xa + k < nw) ? (uint32_t)rowp[xa + k] : 120000u;
                }
                // left -> right
#pragma unroll
                for (int t = 0; t < 2; ++t) {
                    d[t] = 120000u;
#pragma unroll
                    for (int k = 0; k < 8; ++k) if (k < chunk) d[t] = min(d[t] + CELL_W, v[t][k]);
                    e[t] = d[t];
                }
#pragma unroll
                for (int s_ = 1; s_ < 32; s_ <<= 1) {
#pragma unroll
                    for (int t = 0; t < 2; ++t) {
                        const uint32_t o = __shfl_up_sync(0xffffffffu, e[t], s_);
                        if (lane >= s_) e[t] = min(e[t], o + (uint32_t)(s_ * chunk * CELL_W));
                    }
                }
#pragma unroll
                for (int t = 0; t < 2; ++t) {
                    const uint32_t cin = __shfl_up_sync(0xffffffffu, e[t], 1);
                    d[t] = lane == 0 ? 120000u : cin;
#pragma unroll
                    for (int k = 0; k < 8; ++k) if (k < chunk) { d[t] = min(d[t] + CELL_W, v[t][k]); v[t][k] = d[t]; }
                    // right -> left
                    d[t] = 120000u;
#pragma unroll
                    for (int k = 7; k >= 0; --k) if (k < chunk) d[t] = min(d[t] + CELL_W, v[t][k]);
                    e[t] = d[t];
                }
#pragma unroll
                for (int s_ = 1; s_ < 32; s_ <<= 1) {
#pragma unroll
                    for (int t = 0; t < 2; ++t) {
                        const uint32_t o = __shfl_down_sync(0xffffffffu, e[t], s_);
                        if (lane + s_ < 32) e[t] = min(e[t], o + (uint32_t)(s_ * chunk * CELL_W));
                    }
                }
#pragma unroll
                for (int t = 0; t < 2; ++t) {
                    const uint32_t cin = __shfl_down_sync(0xffffffffu, e[t], 1);
                    d[t] = lane == 31 ? 120000u : cin;
                    mx[t] = 0;
#pragma unroll
                    for (int k = 7; k >= 0; --k)
                        if (k < chunk) { d[t] = min(d[t] + CELL_W, v[t][k]); if (xa + k < nw) mx[t] = max(mx[t], d[t]); }
                }
#pragma unroll
                for (int s_ = 16; s_ > 0; s_ >>= 1) {
#pragma unroll
                    for (int t = 0; t < 2; ++t) mx[t] = max(mx[t], __shfl_xor_sync(0xffffffffu, mx[t], s_));
                }
#pragma unroll
                for (int t = 0; t < 2; ++t) {
                    const int cy = cy0 + 8 * t;
                    if (lane == 0 && cy < nh) cellU[cy] = (int)min(mx[t], 60000u) + (CELL_H - 1) + (CELL_W - 1);   // >= max dt of the cell row
                }
            }
        } else {
            for (int cy = c0row + pw * 32 + lane; cy < nh; cy += 256) {      // very wide frames: one thread per cell row
                uint32_t d = 60000;
                for (int cx = 0; cx < nw; ++cx) { d = min(d + CELL_W, (uint32_t)cellD[cy * nw + cx]); cellD[cy * nw + cx] = (uint16_t)min(d, 60000u); }
                d = 60000;
                uint32_t mx = 0;
                for (int cx = nw - 1; cx >= 0; --cx) { d = min(d + CELL_W, (uint32_t)cellD[cy * nw + cx]); mx = max(mx, min(d, 60000u)); }
                cellU[cy] = (int)mx + (CELL_H - 1) + (CELL_W - 1);
            }
        }
        planner_sync();
    }
    dbg_mark(4);

    if (ptid == 0) {
        ws.counts[2 * b] = (int)nsrc;
        ws.counts[2 * b + 1] = (int)nval;
        if (out_counts) { out_counts[2 * b] = (int)nsrc; out_counts[2 * b + 1] = (int)nval; }
        // numpy's IndexError: empty depth_list, or a label beyond its end (tools.py:26)
        if (nval == 0 || nsrc > nval) atomicMin(&ws.status[0], b + fp.frame0);
        if (kind == TASK_WIDE) atomicAdd(&ws.status[1], 1);

        int nt = 0;
        Task* t = st;                 // tasks are built in shared memory and written out by all planner threads
        int* cost = scost;
        auto blank = [&](int knd) {
            Task q;
            q.frame = b; q.lo = 0; q.hi = H; q.r0 = 0; q.r1 = H; q.kind = knd; q.scratch_off = 0; q.fstart = 0;
            q.clo = 0; q.c0 = 0; q.c1 = W; q.sky = -2;
            return q;
        };
        // S = rows handed to k3_sky (their distance is that of row f plus the row offset, their label follows a fixed
        // route down to two base rows); the tiles below cover rows [S, H).
        int S = S0;
        if (plan) {
            const int nwid = fp.narrow_ppl * 32;                 // width of a half-width tile (0: never split)
            int cy = S / CELL_H, scr = 0;
            bool ok = true;
            while (cy < nh && ok) {
                const int r0 = cy * CELL_H;
                int lo = 1 << 30, hi = 0, prev = 0, end = cy, best_lo = 0, best_hi = 0, umax = 0, best_u = 0;
                // strict order: the cell row that holds the base rows S, S+1 of k3_sky is a band (and a full-width task)
                // of its own -- a short scan that the side stream finishes early, so that k3_sky's writes run beside
                // the narrow tiles instead of behind them
                const bool base_band = fp.sky_split && S > 0 && r0 == S;
                for (int c = cy; c < nh; ++c) {
                    lo = min(lo, c * CELL_H - cellU[c]);
                    hi = max(hi, min(H, (c + 1) * CELL_H) + cellU[c]);
                    umax = max(umax, cellU[c]);
                    const int L = max(S, lo), Hh = min(H, hi);      // nothing above S feeds the forward pass
                    const int cst = (Hh - L) + (Hh - r0);
                    // extend while the tile stays under the target cost, while extending is (nearly) free, or while
                    // the band is still short compared with its halo (sparse frames: tall bands, less redundancy)
                    const bool take = c == cy || (!base_band && (nt >= MAXT - 4 || cst <= fp.band_cap || cst - prev <= CELL_H ||
                                                                 (c - cy) * CELL_H < 2 * cellU[c]));
                    if (!take) break;
                    prev = cst; end = c + 1; best_lo = L; best_hi = Hh; best_u = umax;
                }
                Task q = blank(TASK_CHAMFER);
                q.lo = best_lo; q.hi = best_hi; q.r0 = r0; q.r1 = min(H, end * CELL_H);
                q.sky = (S > 0 && r0 == S) ? S : -2;
                // n overlapping narrow tiles when the bound leaves every written pixel's ball inside its tile and the
                // extra columns stay below ~60 % (n * nwid <= 1.6 W)
                int ntile = 0;
                if (nwid > 0 && W > nwid && (W & 3) == 0 && !base_band) {
                    for (int n = 2; n <= fp.max_col_tiles && !ntile; ++n) {
                        if (5 * n * nwid > 8 * W || nt + n > MAXT) break;
                        bool fits = true;                      // every interior tile edge at least best_u away
                        int prev_split = 0;
                        for (int k = 0; k < n && fits; ++k) {
                            const int s0 = (((W - nwid) * k / (n - 1)) & ~3);
                            const int s1 = (((W - nwid) * (k + 1) / (n - 1)) & ~3);
                            const int split = k == n - 1 ? W : ((s1 + s0 + nwid) / 2) & ~3;
                            if ((k > 0 && prev_split - s0 < best_u) || (k < n - 1 && s0 + nwid - split < best_u) ||
                                split <= prev_split) fits = false;
                            prev_split = split;
                        }
                        if (fits) ntile = n;
                    }
                }
                if (ntile) {
                    q.kind = TASK_NARROW;
                    int prev_split = 0;
                    for (int k = 0; k < ntile; ++k) {
                        const int s0 = (((W - nwid) * k / (ntile - 1)) & ~3);           // sub-image start
                        const int s1 = (((W - nwid) * (k + 1) / (ntile - 1)) & ~3);     // next tile's start
                        const int split = k == ntile - 1 ? W : ((s1 + s0 + nwid) / 2) & ~3;        // middle of the overlap
                        q.clo = s0; q.c0 = prev_split; q.c1 = split; q.scratch_off = scr;
                        // halo check (the sizes above guarantee it; keep the planner honest)
                        if ((k > 0 && q.c0 - s0 < best_u) || (k < ntile - 1 && s0 + nwid - split < best_u)) ok = false;
                        scr += (best_hi - best_lo) * fp.narrow_ppl;
                        cost[nt] = prev; t[nt++] = q;
                        prev_split = split;
                    }
                } else {
                    q.scratch_off = scr;
                    scr += (best_hi - best_lo) * fp.wide_ppl;
                    cost[nt] = 2 * prev;                      // twice the work per row step of a narrow tile
                    t[nt++] = q;
                }
                if (scr > fp.scratch_units_per_frame) ok = false;
                cy = end;
            }
            if (!ok) { nt = 0; S = 0; }
        }
        ws.sky[b] = S;
        if (nt == 0) {
            cost[0] = 4 * H;
            t[nt++] = blank(kind);
        }
        snt = nt;
    }
    dbg_mark(5);
    planner_sync();
    // ---- all planner threads: order the tasks (longest first: the block scheduler hands out blocks in index
    // order, slot-major task array), fill in the forward start rows, write the 32 slots of this frame
    {
        const int nt = snt;
        if (ptid < MAXT) {
            Task q;
            int slot = ptid;
            if (ptid < nt) {
                const int c = scost[ptid];
                int rank = 0;
                for (int j = 0; j < nt; ++j) rank += (scost[j] > c) || (scost[j] == c && j < ptid);
                slot = rank;
                q = st[ptid];
                if (plan) {       // rows without any source above them stay unreached in the forward pass: skip them
                    int f = H;
                    for (int w = q.lo >> 5; w < 128 && (w << 5) < H; ++w) {
                        uint32_t m = srcrows[w];
                        if (w == (q.lo >> 5)) m &= ~0u << (q.lo & 31);
                        if (m) { f = min(H, (w << 5) + __ffs(m) - 1); break; }
                    }
                    q.fstart = min(f, q.hi - 1);
                }
                q.scratch_off += b * fp.scratch_units_per_frame;
            } else {
                q.frame = b; q.lo = 0; q.hi = 0; q.r0 = 0; q.r1 = 0; q.kind = TASK_SKIP; q.scratch_off = 0; q.fstart = 0;
                q.clo = 0; q.c0 = 0; q.c1 = W; q.sky = -2;
            }
            ws.tasks[(long)slot * B + b] = q;
        }
    }
    dbg_mark(6);
}

}  // namespace dtfill
