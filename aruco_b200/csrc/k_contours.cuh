// Stage 2a: border extraction (replaces cv::findContours(RETR_LIST, CHAIN_APPROX_NONE),
// src/markerdetector.cpp:510-511, and the length filter at :517).  See ab_trace.cuh for the algorithm.
//   k_scan_starts:  bitwise scan of the tiled packed image for start candidates (one thread per word column x 4 rows)
//   k_trace<false>: one lane per candidate walks its border cycle in both directions; walks alive after 48 iterations
//                   are parked.  k_trace<true> finishes the parked walks and RECORDS the pixels it visits in a per-lane
//                   strip; the Suzuki start of every border with min_len < n < max_len reserves its slice of the point
//                   pool and leaves a contour record, and the warp copies the winner's strip into the slice.
//   k_emit:         re-walks what is not recorded: contours closed by k_trace<false> (2 walkers per contour) and the
//                   first TRACE_PARK_N steps in either direction of the long ones.
#pragma once
#include "ab_device.cuh"

namespace ab {

// one thread per word column x 4 rows of a bit tile (128-bit loads; a warp reads 4 whole tiles = 512 contiguous
// bytes, plus the same rows of the west and east tiles); candidates are appended with ONE atomic per CTA and
// iteration (one per warp put 520 k atomics on the same counter and the kernel waited on their round trips:
// 76 % long-scoreboard stalls in ncu r1o)
__global__ void __launch_bounds__(256) k_scan_starts(Batch b) {
    __shared__ int s_tot[8];
    __shared__ unsigned long long s_base;
    const int ww = (b.W + 31) >> 5;
    const int trows = (b.H + 2 + BIT_TILE - 1) / BIT_TILE;
    const unsigned long long total = (unsigned long long)ww * 8ull * trows * b.B;
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    for (unsigned long long cbase = (unsigned long long)blockIdx.x * blockDim.x; cbase < total;
         cbase += (unsigned long long)gridDim.x * blockDim.x) {  // CTA-uniform trip count: barriers inside
        unsigned long long i = cbase + threadIdx.x;
        uint32_t outer[4] = {0, 0, 0, 0}, hole[4] = {0, 0, 0, 0};
        int wcl = 0, y0 = 0, f = 0, cnt = 0;
        if (i < total) {
            // 32-bit index arithmetic (the host checks total < 2^32): four 64-bit divisions per item were ~half of this
            // kernel's instructions
            const unsigned i32 = (unsigned)i, row_items = 8u * (unsigned)ww, frame_items = row_items * (unsigned)trows;
            f = (int)(i32 / frame_items);
            const unsigned rem = i32 - (unsigned)f * frame_items;
            const int ty = (int)(rem / row_items);
            const unsigned r2 = rem - (unsigned)ty * row_items;
            const int g = (int)(r2 & 7u);
            wcl = (int)(r2 >> 3);
            y0 = ty * BIT_TILE + 4 * g - 1;  // image row of the first of the 4 rows (padded row - 1)
            const uint32_t* tile = b.bits + (size_t)f * b.bits_words + ((size_t)ty * b.wpr + (wcl + BIT_PAD)) * BIT_TILE;
            const uint4 c4 = *reinterpret_cast<const uint4*>(tile + 4 * g);
            const uint4 w4 = *reinterpret_cast<const uint4*>(tile - BIT_TILE + 4 * g);
            const uint4 e4 = *reinterpret_cast<const uint4*>(tile + BIT_TILE + 4 * g);
            uint32_t cu = 0, wu = 0, eu = 0;  // the row above the first row
            if (g > 0) {
                cu = tile[4 * g - 1];
                wu = tile[4 * g - 1 - BIT_TILE];
                eu = tile[4 * g - 1 + BIT_TILE];
            } else if (ty > 0) {
                const uint32_t* up = tile - (size_t)b.wpr * BIT_TILE + (BIT_TILE - 1);
                cu = up[0];
                wu = up[-BIT_TILE];
                eu = up[BIT_TILE];
            }
            const uint32_t c[5] = {cu, c4.x, c4.y, c4.z, c4.w}, w[5] = {wu, w4.x, w4.y, w4.z, w4.w}, e[5] = {eu, e4.x, e4.y, e4.z, e4.w};
#pragma unroll
            for (int k = 0; k < 4; k++) {
                uint32_t cur = c[k + 1], west = (cur << 1) | (w[k + 1] >> 31);
                uint32_t uu = c[k], uw = (uu << 1) | (w[k] >> 31), ue = (uu >> 1) | (e[k] << 31);
                outer[k] = cur & ~west & ~uu & ~uw & ~ue;  // fg with W, N, NW, NE background
                hole[k] = ~cur & west & uu;                // bg with W and N foreground
                cnt += __popc(outer[k]) + __popc(hole[k]);
            }
        }
        int incl = cnt;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            int v = __shfl_up_sync(0xFFFFFFFFu, incl, d);
            if (lane >= d) incl += v;
        }
        if (lane == 31) s_tot[warp] = incl;
        __syncthreads();
        int before = 0, tot = 0;  // candidates of the warps before this one / of the whole CTA
#pragma unroll
        for (int w = 0; w < 8; w++) {
            const int v = s_tot[w];
            before += w < warp ? v : 0;
            tot += v;
        }
        if (threadIdx.x == 0 && tot) s_base = atomicAdd(&b.cnt->n_starts, (unsigned long long)tot);
        __syncthreads();
        if (tot == 0) continue;
        const unsigned long long cta_base = s_base;
        if (cta_base + (unsigned long long)tot > b.cap_starts) {
            if (threadIdx.x == 0) atomicOr(&b.cnt->err, ERR_STARTS_OVERFLOW);
            continue;
        }
        unsigned long long o = cta_base + (unsigned long long)(before + incl - cnt);
#pragma unroll
        for (int k = 0; k < 4; k++) {
            uint32_t m = outer[k];
            const uint32_t xb = (uint32_t)(32 * wcl), y = (uint32_t)(y0 + k);
            while (m) {
                int j = __ffs((int)m) - 1;
                m &= m - 1;
                AB_BOUND(o < b.cap_starts);
                b.starts[o++] = make_uint2((uint32_t)f, (xb + j) | (y << 16));
            }
            m = hole[k];
            while (m) {
                int j = __ffs((int)m) - 1;
                m &= m - 1;
                AB_BOUND(o < b.cap_starts);
                b.starts[o++] = make_uint2((uint32_t)f | 0x80000000u, (xb + j) | (y << 16));
            }
        }
    }
}

// Lane-scheduled walker.  Every lane owns one start candidate at a time and is refilled from a global work
// counter as soon as it finishes, so a warp never idles behind its longest contour (border lengths range
// from 2 to max_len).  The walk is the bidirectional search of find_start_bidir (ab_trace.cuh), executed
// STEPS at a time; the Suzuki start of a border with min_len < n < max_len reserves its slice of the point
// pool and leaves a contour record -- the points themselves are written by k_emit.
//
// Two-level scheduling: border lengths are extremely skewed (thousands of 2..30-step speckle walks per frame,
// a few hundred walks of 300..3800 steps).  A walk that is still alive after LONG_T steps is parked in a queue
// (full walker state) and its lane is refilled; k_trace<true> then runs the parked walks to completion in
// densely populated warps.  Without this, the long walks end up one or two per warp and the kernel spends
// most of its time issuing instructions for ~9 of 32 lanes (ncu r1e).
constexpr int TRACE_LONG_T = 48;
constexpr int TRACE_STEPS = 8, TRACE_STEPS_LONG = 8;  // iterations per round of k_trace<false> / k_trace<true>
// iterations a walk has made when k_trace<false> parks it: lanes are refilled only between rounds of TRACE_STEPS
// iterations, so the count is the first multiple of the round length that reaches the parking threshold
constexpr int TRACE_PARK_N = (TRACE_LONG_T + TRACE_STEPS - 1) / TRACE_STEPS * TRACE_STEPS;
static_assert(TRACE_PARK_N % 2 == 0 && TRACE_STEPS_LONG % 2 == 0, "paired strip stores need even rounds");

// `s` is the start state of a start candidate (table flags e): does its trigger scan before key0?
// (raster positions fit 32 bits: W, H <= 16384)
__device__ __forceinline__ bool smaller_trigger(uint32_t e, const WalkState& s, int W, int64_t key0) {
    const uint32_t k = (uint32_t)(s.y * W + s.x), k0 = (uint32_t)key0;
    return ((e & WALK_TRIG_OUTER) && k < k0) || ((e & WALK_TRIG_HOLE) && k + 1u < k0);
}

template <bool LONG>
__global__ void __launch_bounds__(128) k_trace(Batch b) {
    constexpr int STEPS = LONG ? TRACE_STEPS_LONG : TRACE_STEPS;
    const unsigned FULL = 0xFFFFFFFFu;
    const int lane = threadIdx.x & 31;
    unsigned long long n_items;
    if (LONG) {
        n_items = b.cnt->n_long;
        if (n_items > b.cap_long) n_items = b.cap_long;
    } else {
        n_items = b.cnt->n_starts;
        if (n_items > b.cap_starts) return;  // overflow already flagged by k_scan_starts; the list has holes
    }
    unsigned int* work = LONG ? &b.cnt->long_work : &b.cnt->trace_work;
    bool active = false, exhausted = false, nodefer = LONG;
    BitImage im = b.bit_image(0);
    TraceStart st{0, 0, 0, 0};
    WalkState fw{0, 0, 0}, bw{0, 0, 0};
    uint32_t e_fw = 0, type_bit = 0;  // e_fw: forward table entry of the current forward state
    const uint8_t* __restrict__ lut_fw = b.walk_lut;
    const uint8_t* __restrict__ lut_bw = b.walk_lut + WALK_LUT_SIZE;
    int nf = 0, ng = 0, frame = 0;
    // LONG only: entry k of the lane's strip = (pixel of the forward walker after TRACE_PARK_N + 1 + k steps, pixel of the
    // backward walker after as many) = points TRACE_PARK_N + 1 + k and n - TRACE_PARK_N - 1 - k of the contour.  Losers
    // record for nothing (8 bytes per iteration); winners save the second walk over the border that k_emit_long used to
    // make (one dependent L1/L2 round trip per point, 0.5 ms per 256 4K frames).
    const unsigned gid = blockIdx.x * blockDim.x + threadIdx.x;
    uint2* const rec = LONG ? b.trace_rec + (size_t)gid * b.rec_half : nullptr;
    uint32_t cp_off = 0;
    uint2 rec_prev = make_uint2(0u, 0u);
    int cp_len = 0;  // > 0: this lane's walk closed a kept contour whose strip is still to be copied
    for (;;) {
        unsigned idle = __ballot_sync(FULL, !active && !exhausted);
        if (idle) {
            unsigned base = 0;
            int leader = __ffs((int)idle) - 1;
            if (lane == leader) base = atomicAdd(work, (unsigned)__popc(idle));
            base = __shfl_sync(FULL, base, leader);
            if (!active && !exhausted) {
                unsigned long long i = (unsigned long long)base + (unsigned)__popc(idle & ((1u << lane) - 1u));
                if (i >= n_items) {
                    exhausted = true;
                } else if (LONG) {
                    const LongRec q = b.longq[i];
                    frame = (int)(q.frame & 0x7FFFFFFFu);
                    type_bit = q.frame & 0x80000000u;
                    im = b.bit_image(frame);
                    st.key = q.key;
                    st.x = (int)(q.sxy & 0xFFFFu);
                    st.y = (int)(q.sxy >> 16);
                    st.b = (int)((q.dirs >> 8) & 7u);
                    fw = WalkState{(int)(q.fxy & 0xFFFFu), (int)(q.fxy >> 16), (int)(q.dirs & 7u)};
                    bw = WalkState{(int)(q.bxy & 0xFFFFu), (int)(q.bxy >> 16), (int)((q.dirs >> 4) & 7u)};
                    nf = (int)q.nf;
                    ng = (int)q.ng;
                    AB_BOUND(nf == TRACE_PARK_N && ng == TRACE_PARK_N);
                    e_fw = lut_fw[window9(im, fw.x, fw.y) | ((uint32_t)fw.b << 9)];
                    active = true;
                } else {
                    uint2 rec = b.starts[i];
                    frame = (int)(rec.x & 0x7FFFFFFFu);
                    type_bit = rec.x & 0x80000000u;
                    im = b.bit_image(frame);
                    if (make_start(im, (int)(rec.x >> 31), (int)(rec.y & 0xFFFFu), (int)(rec.y >> 16), st)) {
                        fw = WalkState{st.x, st.y, st.b};
                        bw = fw;
                        e_fw = lut_fw[window9(im, fw.x, fw.y) | ((uint32_t)fw.b << 9)];
                        nf = ng = 0;
                        nodefer = false;
                        active = true;
                    }  // else: isolated pixel, a 1-point contour that is never kept
                }
            }
        }
        if (__ballot_sync(FULL, active) == 0) {
            if (__ballot_sync(FULL, !exhausted) == 0) break;
            continue;
        }
        if (active) {
            for (int r = 0; r < STEPS; r++) {
                bool closed = false, dead = false;
                // both walkers step first so that their neighbourhood loads are in flight together (the two
                // dependent load rounds per iteration were the latency floor of long walks); the backward step
                // is only COMMITTED if the forward step neither closed the cycle nor hit a smaller start
                const WalkState bw0 = bw;
                {
                    const int d = (int)(e_fw & 7u);
                    fw.x += step_dx(d);
                    fw.y += step_dy(d);
                    fw.b = (d + 4) & 7;
                }
                const uint32_t w_f = window9(im, fw.x, fw.y);
                WalkState bw1{bw0.x + step_dx(bw0.b), bw0.y + step_dy(bw0.b), 0};
                if (LONG) {  // both pixels are known before the step tables answer: the store is off the dependent chain
                    AB_BOUND(nf >= TRACE_PARK_N && (unsigned)(nf - TRACE_PARK_N) < b.rec_half);
                    // two iterations per 16-byte store (one 8-byte store per iteration: k_trace<true> 0.93 instead of 0.77 ms):
                    // a round starts at an even entry (TRACE_PARK_N and the round length are even), so the parity of r is
                    // the parity of the entry; a walk that closes on an even entry flushes its half below.  Plain stores
                    // and plain loads: st.cg / ld.cg were measured and are no faster or much slower (profiles/README.md)
                    const uint2 cur = make_uint2((uint32_t)fw.x | ((uint32_t)fw.y << 16), (uint32_t)bw1.x | ((uint32_t)bw1.y << 16));
                    if (r & 1) *reinterpret_cast<uint4*>(rec + (nf - TRACE_PARK_N - 1)) = make_uint4(rec_prev.x, rec_prev.y, cur.x, cur.y);
                    else rec_prev = cur;
                }
                const uint32_t w_q = window9(im, bw1.x, bw1.y);
                e_fw = lut_fw[w_f | ((uint32_t)fw.b << 9)];
                const uint32_t e_bw = lut_bw[w_q | ((uint32_t)((bw0.b + 4) & 7) << 9)];
                bw1.b = (int)(e_bw & 7u);
                nf++;
                if (same_state(fw, bw0)) {
                    closed = true;
                } else if ((e_fw & (WALK_TRIG_OUTER | WALK_TRIG_HOLE)) && smaller_trigger(e_fw, fw, im.W, st.key)) {
                    dead = true;
                } else {
                    bw = bw1;
                    ng++;
                    if (same_state(fw, bw)) closed = true;
                    else if ((e_bw & (WALK_TRIG_OUTER | WALK_TRIG_HOLE)) && smaller_trigger(e_bw, bw, im.W, st.key)) dead = true;
                    else if (nf + ng >= b.max_len) dead = true;  // too long: dropped by :517 anyway
                }
                if (closed) {
                    const int len = nf + ng;
                    if (len > b.min_len && len < b.max_len) {  // src/markerdetector.cpp:517
                        unsigned int ci = atomicAdd(&b.cnt->n_contours, 1u);
                        unsigned long long off = atomicAdd(&b.cnt->pool_used, (unsigned long long)len);
                        if (ci >= b.cap_contours) {
                            atomicOr(&b.cnt->err, ERR_CONTOURS_OVERFLOW);
                        } else if (off + (unsigned long long)len > b.cap_pool) {
                            atomicOr(&b.cnt->err, ERR_POOL_OVERFLOW);
                            b.contours[ci] = ContourRec{(uint32_t)frame | type_bit, 0u, 0u, (uint32_t)st.key};
                        } else if (!LONG) {
                            b.contours[ci] = ContourRec{(uint32_t)frame | type_bit, (uint32_t)off, (uint32_t)len, (uint32_t)st.key};
                        } else {
                            b.contours[ci] = ContourRec{(uint32_t)frame | type_bit | CONTOUR_LONG, (uint32_t)off, (uint32_t)len, (uint32_t)st.key};
                            cp_off = (uint32_t)off;
                            cp_len = len;
                            if (!(r & 1)) rec[nf - 1 - TRACE_PARK_N] = rec_prev;
                        }
                    }
                    active = false;
                    break;
                }
                if (dead) {
                    active = false;
                    break;
                }
            }
            if (!LONG && active && !nodefer && nf >= TRACE_LONG_T) {
                unsigned int qi = atomicAdd(&b.cnt->n_long, 1u);
                if (qi < b.cap_long) {
                    LongRec q;
                    q.frame = (uint32_t)frame | type_bit;
                    q.key = (uint32_t)st.key;
                    q.sxy = (uint32_t)st.x | ((uint32_t)st.y << 16);
                    q.fxy = (uint32_t)fw.x | ((uint32_t)fw.y << 16);
                    q.bxy = (uint32_t)bw.x | ((uint32_t)bw.y << 16);
                    q.dirs = (uint32_t)fw.b | ((uint32_t)bw.b << 4) | ((uint32_t)st.b << 8);
                    q.nf = (uint32_t)nf;
                    q.ng = (uint32_t)ng;
                    AB_BOUND(qi < b.cap_long);
                    b.longq[qi] = q;
                    active = false;
                } else {
                    nodefer = true;  // queue full: finish this walk in place (correct, just slower)
                }
            }
        }
        if (LONG) {  // winners of this round: the warp copies each strip into its slice of the pool, 32 points at a time
            __syncwarp();  // the strips were written by their own lanes
            unsigned cpm = __ballot_sync(FULL, cp_len > 0);
            while (cpm) {
                const int s = __ffs((int)cpm) - 1;
                cpm &= cpm - 1;
                const int n = __shfl_sync(FULL, cp_len, s);
                const int f = __shfl_sync(FULL, nf, s) - TRACE_PARK_N, g = __shfl_sync(FULL, ng, s) - TRACE_PARK_N;
                uint32_t* dst = b.pool + __shfl_sync(FULL, cp_off, s);
                const uint2* src = b.trace_rec + (size_t)(gid - (unsigned)lane + (unsigned)s) * b.rec_half;
                AB_BOUND(f >= 1 && g >= 0 && g <= f && n == f + g + 2 * TRACE_PARK_N);
                constexpr int CU = 8;  // loads in flight per lane: the copy holds up the other 31 walks of the warp
                for (int k0 = lane; k0 < f; k0 += 32 * CU) {
                    uint2 v[CU];
#pragma unroll
                    for (int u = 0; u < CU; u++)
                        if (k0 + 32 * u < f) v[u] = src[k0 + 32 * u];
#pragma unroll
                    for (int u = 0; u < CU; u++) {
                        const int k = k0 + 32 * u;
                        if (k < f) {
                            dst[TRACE_PARK_N + 1 + k] = v[u].x;
                            if (k < g) dst[n - TRACE_PARK_N - 1 - k] = v[u].y;
                        }
                    }
                }
            }
            cp_len = 0;
        }
    }
}

// Writes the ordered points of every kept contour.  Two work items per contour: one walks forwards from the
// start and fills the first half, the other walks backwards and fills the second half from the end (the
// successor function is a permutation, so the predecessor walk visits the same cycle in reverse).  Lane
// scheduled like k_trace.
__global__ void __launch_bounds__(128) k_emit(Batch b) {
    constexpr int STEPS = 16;
    const unsigned FULL = 0xFFFFFFFFu;
    const int lane = threadIdx.x & 31;
    unsigned int ncont = b.cnt->n_contours;
    if (ncont > b.cap_contours) ncont = b.cap_contours;
    const unsigned int n_items = 2u * ncont;
    bool active = false, exhausted = false, backward = false;
    BitImage im = b.bit_image(0);
    WalkState w{0, 0, 0};
    uint32_t nb = 0;
    int remaining = 0;
    uint32_t* out = nullptr;
    for (;;) {
        unsigned idle = __ballot_sync(FULL, !active && !exhausted);
        if (idle) {
            unsigned base = 0;
            int leader = __ffs((int)idle) - 1;
            if (lane == leader) base = atomicAdd(&b.cnt->emit_work, (unsigned)__popc(idle));
            base = __shfl_sync(FULL, base, leader);
            if (!active && !exhausted) {
                unsigned i = base + (unsigned)__popc(idle & ((1u << lane) - 1u));
                if (i >= n_items) {
                    exhausted = true;
                } else {
                    // items [0, ncont) walk forwards, [ncont, 2 ncont) backwards: warps stay homogeneous, so a round
                    // costs one dependent load round trip instead of two (forward lanes, then backward lanes)
                    const ContourRec rec = b.contours[i < ncont ? i : i - ncont];
                    const int n = (int)rec.n;
                    if (n > 0) {
                        im = b.bit_image((int)(rec.frame & CONTOUR_FRAME_MASK));
                        TraceStart st;
                        make_start(im, (int)(rec.frame >> 31), (int)(rec.key % (uint32_t)b.W), (int)(rec.key / (uint32_t)b.W), st);
                        w = WalkState{st.x, st.y, st.b};
                        // a long contour (n > 2 TRACE_PARK_N) only lacks the points walked before it was parked: 0 .. PARK_N
                        // and n-1 .. n-PARK_N; the others are walked whole, half from either end
                        const bool lng = (rec.frame & CONTOUR_LONG) != 0u;
                        const int h0 = lng ? TRACE_PARK_N + 1 : (n + 1) >> 1;
                        backward = i >= ncont;
                        if (!backward) {
                            out = b.pool + rec.off;  // positions 0 .. h0-1, ascending
                            remaining = h0;
                            nb = neighbours8(im, w.x, w.y);
                        } else {
                            out = b.pool + rec.off + n - 1;  // positions n-1 .. h0 (long: n - PARK_N), descending
                            remaining = lng ? TRACE_PARK_N : n - h0;
                        }
                        active = remaining > 0;
                    }
                }
            }
        }
        if (__ballot_sync(FULL, active) == 0) {
            if (__ballot_sync(FULL, !exhausted) == 0) break;
            continue;
        }
        if (active) {
            if (!backward) {
                for (int r = 0; r < STEPS; r++) {
                    AB_BOUND(out >= b.pool && out < b.pool + b.cap_pool);
                    *out++ = (uint32_t)w.x | ((uint32_t)w.y << 16);
                    if (--remaining == 0) {
                        active = false;
                        break;
                    }
                    walk_forward(w, nb);
                    nb = neighbours8(im, w.x, w.y);
                }
            } else {
                for (int r = 0; r < STEPS; r++) {
                    walk_backward(im, w);
                    AB_BOUND(out >= b.pool && out < b.pool + b.cap_pool);
                    *out-- = (uint32_t)w.x | ((uint32_t)w.y << 16);
                    if (--remaining == 0) {
                        active = false;
                        break;
                    }
                }
            }
        }
    }
}

}  // namespace ab
