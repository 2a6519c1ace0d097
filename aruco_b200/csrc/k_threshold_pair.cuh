// Adaptive threshold, second generation (same arithmetic as k_threshold_adaptive; k_threshold.cuh states it).
//
// ncu r1d/r1g: k_threshold_fast is issue bound on the ALU pipe at ~27 instructions per pixel while moving only
// 22 % of what HBM could.  This kernel cuts the instruction count ~3x by never unpacking:
//   * a thread owns 4 columns at c and 4 columns at c + HO (half a tile further right); the two are carried as the
//     two 16-bit lanes of one register from the load to the comparison.  Lane partners are never neighbours, so
//     the horizontal window needs no byte shuffling: S(x+1) = S(x) - w[x-R] + w[x+R+1] is ONE 3-input add for 2 pixels,
//   * vertical sums:  V += P_new - P_old  (one add per 2 pixels, the K most recent packed rows live in registers),
//   * published with one 16-byte shared store per thread and row (double buffered, one barrier per row), read back
//     with 16-byte loads,
//   * mean test  S >= K^2 (src + idelta) - (K^2-1)/2  evaluated for both lanes by one IMAD:
//     D = S + (0x8000 - cst) - K^2 * src  has bit 15 of a lane set  <=>  the pixel is foreground,
//   * PRMT with sign replication turns the lane sign bits into 0x00/0xFF output bytes (4 PRMT per 8 pixels),
//   * the 1-bit packed copy is assembled with three shuffles for both halves together.
// Valid while K^2 * 255 + |cst| < 2^15 (K <= 11 with the usual small deltas); otherwise the dispatcher falls back to
// k_threshold_fast / k_threshold_adaptive.
#pragma once
#include "k_threshold_fast.cuh"

namespace ab {

constexpr int THP_RH = 128;  // output rows per CTA before rounding down to whole double turns of the ring

template <uint32_t SEL>
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "n"(SEL));  // default mode: selector bit 3 replicates the sign
    return d;
}

__device__ __forceinline__ uint32_t prmt_r(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ void lds128(uint32_t addr, uint32_t& x, uint32_t& y, uint32_t& z, uint32_t& w) {
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(x), "=r"(y), "=r"(z), "=r"(w) : "r"(addr) : "memory");
}

// Requires W % 4 == 0 and 4-byte aligned source rows (the dispatcher checks): a thread's 4 columns are then either all
// inside the image, all left of it or all right of it, and the replicated border is a PRMT selector, not a branch.
template <int K, int TO>
__global__ void __launch_bounds__(TO + 32, 1) k_threshold_pair(ThrArgs a) {
    constexpr int R = K / 2, R4 = (R + 3) & ~3, HT = R4 / 4, NV = 4 + 2 * R4, HO = 4 * TO, TW = 2 * HO, CSW = HO + 2 * R4, K2 = K * K;
    constexpr uint32_t BUF_BYTES = CSW * 4;
    constexpr int NT = TO + 2 * HT;              // working threads
    constexpr int DEPTH = 8;                     // source rows in flight (cp.async groups)
    constexpr uint32_t STAGE_ROW = NT * 8;       // bytes of one staged row: 2 words per thread
    constexpr int RH = (THP_RH / (2 * K)) * (2 * K);  // rows per CTA: whole double turns of the ring, so the unrolled loop has no exits
    __shared__ __align__(16) uint32_t cs[4][CSW];  // two buffers of two rows
    __shared__ __align__(16) uint2 stage[DEPTH][NT];  // ncu r1j: with loads held in registers two of the K unrolled steps
                                                      // waited ~1 row on the scoreboard; cp.async groups decouple them
    const int t = threadIdx.x;
    if (t >= NT) return;  // spare lanes of the halo warp
    const int X0 = blockIdx.x * TW, y0 = blockIdx.y * RH, f = blockIdx.z;
    const bool is_out = t < TO;
    // ci: index into a row of cs.  cs[ci] = (V[X0 - R4 + ci], V[X0 + HO - R4 + ci])
    const int ci = is_out ? R4 + 4 * t : (t < TO + HT ? 4 * (t - TO) : R4 + HO + 4 * (t - TO - HT));
    const int ca = X0 - R4 + ci, cb = ca + HO;
    // replicated border: load the nearest in-image word and let the packing PRMT pick byte 0 (left) or 3 (right)
    uint32_t sel[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const uint32_t ja = ca < 0 ? 0u : (ca >= a.W ? 3u : (uint32_t)j), jb = 4u + (cb >= a.W ? 3u : (uint32_t)j);
        sel[j] = ja | (ja << 4) | (jb << 8) | (jb << 12);
    }
    const int nout = min(RH, a.H - y0);  // rows below the image are computed (clamped loads) but not stored
    int yraw = y0 - R;  // source row of the next ring step, before clamping to the image
    const uint8_t* src = a.grey + (size_t)f * a.grey_frame + (size_t)min(max(yraw, 0), a.H - 1) * a.grey_row;
    const uint8_t* pa = src + min(max(ca, 0), a.W - 4);
    const uint8_t* pb = src + min(cb, a.W - 4);
    const bool ok_a = is_out && ca < a.W, ok_b = is_out && cb < a.W;
    const size_t fo = (size_t)f * a.out_mul + a.out_off;
    uint8_t* orow = a.thres + fo * a.W * a.H + (size_t)y0 * a.W + ca;
    uint32_t* brow = a.bits + fo * a.bits_words + bit_word_index(a.wpr, BIT_PAD + (X0 >> 5) + (t >> 3), y0);
    int btr = (y0 + 1) & 31;  // row inside the bit tile
    const int bjump = a.wpr * BIT_TILE - (BIT_TILE - 1);
    const bool word_a = ok_a && (t & 7) == 0, word_b = ok_b && (t & 7) == 0;
    const int cst = K2 * a.idelta - (K2 - 1) / 2;  // S >= K2*src + cst  <=>  src - mean <= -idelta
    const uint32_t GC = (uint32_t)((0x8000 - cst) & 0xFFFF) * 0x00010001u;
    const uint32_t M = 0x00FF00FFu;
    const uint32_t s_base = (uint32_t)__cvta_generic_to_shared(&cs[0][0]);
    const uint32_t s_wr = s_base + 4u * ci, s_rd = s_base + 4u * (ci - R4);
    const int nib_shift = 4 * (t & 3);
    uint32_t boff = 0;

    const int nrows = nout + 2 * R;  // ring steps this CTA consumes
    const uint32_t s_stage = (uint32_t)__cvta_generic_to_shared(&stage[0][t]);
    uint32_t soff = 0;
    int issued = 0;
    auto issue_row = [&](uint32_t off) {  // async copy of the next source row into stage slot `off`
        if (issued < nrows) {
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s_stage + off), "l"(pa) : "memory");
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s_stage + off + 4u), "l"(pb) : "memory");
            const size_t inc = ((unsigned)yraw < (unsigned)(a.H - 1)) ? a.grey_row : (size_t)0;
            pa += inc;
            pb += inc;
            yraw++;
        }
        issued++;
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto load_row = [&]() -> uint2 {  // oldest staged row; its slot is refilled with the row DEPTH steps ahead
        uint2 p;
        asm volatile("cp.async.wait_group %0;" ::"n"(DEPTH - 1) : "memory");
        asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(p.x), "=r"(p.y) : "r"(s_stage + soff) : "memory");
        issue_row(soff);
        soff = soff + STAGE_ROW == DEPTH * STAGE_ROW ? 0u : soff + STAGE_ROW;
        return p;
    };
#pragma unroll
    for (int d = 0; d < DEPTH; d++) issue_row(d * STAGE_ROW);

    uint32_t ring[K][4];
#pragma unroll
    for (int j = 0; j < K; j++) ring[j][0] = ring[j][1] = ring[j][2] = ring[j][3] = 0u;
    uint32_t V0 = 0u, V1 = 0u, V2 = 0u, V3 = 0u;
    // one ring step: the packed row enters slot j, the row K steps older leaves the vertical sums
    auto accumulate = [&](uint32_t* slot) {
        const uint2 p = load_row();
        const uint32_t P0 = prmt_r(p.x, p.y, sel[0]) & M, P1 = prmt_r(p.x, p.y, sel[1]) & M, P2 = prmt_r(p.x, p.y, sel[2]) & M,
                       P3 = prmt_r(p.x, p.y, sel[3]) & M;
        V0 = V0 + P0 - slot[0];
        V1 = V1 + P1 - slot[1];
        V2 = V2 + P2 - slot[2];
        V3 = V3 + P3 - slot[3];
        slot[0] = P0;
        slot[1] = P1;
        slot[2] = P2;
        slot[3] = P3;
    };
#pragma unroll
    for (int j = 0; j < 2 * R; j++) accumulate(ring[j]);
    // horizontal window sums, comparison and stores of one output row whose column sums sit at shared offset `rd`
    auto emit_row = [&](uint32_t rd, const uint32_t* c, bool row_ok) {
        uint32_t w[NV];
#pragma unroll
        for (int q = 0; q < NV / 4; q++) lds128(rd + 16u * q, w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
        uint32_t S0 = GC;
#pragma unroll
        for (int d = R4 - R; d <= R4 + R; d++) S0 += w[d];
        const uint32_t S1 = S0 - w[R4 - R] + w[R4 + R + 1];
        const uint32_t S2 = S1 - w[R4 - R + 1] + w[R4 + R + 2];
        const uint32_t S3 = S2 - w[R4 - R + 2] + w[R4 + R + 3];
        const uint32_t D0 = S0 - (uint32_t)K2 * c[0], D1 = S1 - (uint32_t)K2 * c[1], D2 = S2 - (uint32_t)K2 * c[2],
                       D3 = S3 - (uint32_t)K2 * c[3];
        // sign bytes (bits 15 / 31) -> 0x00 / 0xFF output bytes of the two halves
        const uint32_t L1 = prmt<0xFBD9>(D0, D1), L2 = prmt<0xFBD9>(D2, D3);
        const uint32_t out_a = prmt<0x5410>(L1, L2), out_b = prmt<0x7632>(L1, L2);
        if (ok_a && row_ok) *reinterpret_cast<uint32_t*>(orow) = out_a;
        if (ok_b && row_ok) *reinterpret_cast<uint32_t*>(orow + HO) = out_b;
        const uint32_t nib_a = ok_a ? ((out_a & 0x08040201u) * 0x01010101u) >> 24 : 0u;
        const uint32_t nib_b = ok_b ? ((out_b & 0x08040201u) * 0x01010101u) >> 24 : 0u;
        // 8 threads make one 32-bit word per half: two levels carry both halves in one register
        uint32_t x = (nib_a | (nib_b << 16)) << nib_shift;
        x |= __shfl_xor_sync(0xFFFFFFFFu, x, 1);
        x |= __shfl_xor_sync(0xFFFFFFFFu, x, 2);
        const uint32_t y = __shfl_xor_sync(0xFFFFFFFFu, x, 4);
        if (word_a && row_ok) brow[0] = prmt<0x5410>(x, y);
        if (word_b && row_ok) brow[(HO / 32) * BIT_TILE] = prmt<0x7632>(x, y);
        orow += a.W;
        brow += btr == 31 ? bjump : 1;
        btr = (btr + 1) & 31;
    };
    // two rows per barrier (ncu r1p: 23 % of the stall samples sat on the per-row barrier, 24 % on the shared loads and
    // shuffles behind it): the column sums of rows A and B are published together, then both rows are finished with
    // twice the independent work in flight.  Row B's ring slot is never row A's centre slot (they differ by R mod K).
    for (int o = 0; o < nout; o += 2 * K) {
#pragma unroll
        for (int jj = 0; jj < 2 * K; jj += 2) {
            accumulate(ring[(2 * R + jj) % K]);
            sts128(s_wr + boff, V0, V1, V2, V3);
            accumulate(ring[(2 * R + jj + 1) % K]);
            sts128(s_wr + boff + BUF_BYTES, V0, V1, V2, V3);
            __syncthreads();
            if (is_out) {
                emit_row(s_rd + boff, ring[(R + jj) % K], o + jj < nout);
                emit_row(s_rd + boff + BUF_BYTES, ring[(R + jj + 1) % K], o + jj + 1 < nout);
            }
            boff = 2 * BUF_BYTES - boff;
        }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
}

// host-side dispatch: returns false when (K, idelta) is outside the 15-bit lane budget
inline bool launch_threshold_pair(const ThrArgs& a, int B, cudaStream_t st) {
    const int K2 = a.k * a.k;
    const long long cst = (long long)K2 * a.idelta - (K2 - 1) / 2;
    if (a.k < 3 || a.k > 11 || !(a.k & 1) || !a.aligned4 || (a.W & 3) || a.W < 4) return false;
    if (K2 * 255LL + (cst < 0 ? -cst : cst) >= 0x8000) return false;
    // tile width 8*TO columns: pick the TO that wastes the fewest columns, the widest on a tie
    int best_to = 128, best_pad = 1 << 30;
    for (int to = 128; to >= 64; to -= 32) {
        int tw = 8 * to, pad = (a.W + tw - 1) / tw * tw;
        if (pad < best_pad) best_pad = pad, best_to = to;
    }
    const int tw = 8 * best_to;
    const int rh = (THP_RH / (2 * a.k)) * (2 * a.k);
    dim3 grid((a.W + tw - 1) / tw, (a.H + rh - 1) / rh, B);
#define AB_THP_TO(KK, TT)                                        \
    if (best_to == TT) {                                         \
        k_threshold_pair<KK, TT><<<grid, TT + 32, 0, st>>>(a);  \
        return true;                                             \
    }
#define AB_THP_CASE(KK) \
    case KK:            \
        AB_THP_TO(KK, 128) AB_THP_TO(KK, 96) AB_THP_TO(KK, 64) return false;
    switch (a.k) {
        AB_THP_CASE(3)
        AB_THP_CASE(5)
        AB_THP_CASE(7)
        AB_THP_CASE(9)
        AB_THP_CASE(11)
        default:
            return false;
    }
#undef AB_THP_CASE
#undef AB_THP_TO
}

}  // namespace ab
