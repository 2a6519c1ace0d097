// Adaptive threshold, third generation: the arithmetic of k_threshold_pair (lane-paired 16-bit sums, see there) with
// the source tile staged by the TMA engine and the image-border logic taken out of the row loop.
//
// ncu r1x on k_threshold_pair<7,96>: 930 M warp-instructions for 2.12 G pixels, 112 registers, issue 57 %; ~17 % of the
// loop body was clamp / predicate logic only border tiles need and every thread spent ~10 instructions per row on the
// cp.async ring (two LDGSTS, pointer bumps, row clamp, group bookkeeping).  Here
//   * ONE elected thread per CTA issues `cp.async.bulk.tensor.3d` copies, one per source row, into a ring of row groups
//     in shared memory; completion is signalled on an mbarrier per group (expect_tx = rows x row bytes).  The replicated
//     top/bottom border is a clamped row COORDINATE at issue time, not a per-thread test; rows left/right of the image
//     arrive zero-filled and are never used: halo threads read the nearest in-image word and replicate its edge byte with
//     the same packing PRMT that every thread executes anyway (selectors in registers),
//   * tiles divide the image width exactly (the dispatcher picks TO accordingly), so there is no column predicate at all;
//     the row predicate exists only in the instantiation used for the last, partial row group of the bottom CTA row,
//   * a thread reads its two source words with immediate-offset shared loads (row slots are compile-time inside the
//     unrolled 2K-row body).
// Shared memory per CTA: NG x 2K staged rows of TW + 32 bytes (pitch rounded up to 128) + the 4 column-sum rows:
// 31.4 KB for K = 7, TO = 96.
#pragma once
#include <cuda.h>
#include "k_threshold_pair.cuh"

namespace ab {

// row groups in flight (r2c: 2 -> 1.33 ms, 3 -> 1.34 ms, 4 -> 1.57 ms; shared memory taken here is L1 taken from co-running kernels)
constexpr int THT_NG = 2;
constexpr int THT_RH = 128;  // output rows per CTA before rounding down to whole groups
// wide kernel: rows per TMA group (r2q, K = 21: 8 -> 0.56 ms, 10 -> 0.61, 14 -> 0.62 per 64 frames; 43 instead of 54 KB per CTA)
constexpr int THW_GR = 8;

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "AB_MBAR_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra AB_MBAR_DONE;\n"
        "bra AB_MBAR_WAIT;\n"
        "AB_MBAR_DONE:\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}
// one source row (box = row bytes x 1 x 1 of the [B][H][W/4] u32 tensor) -> shared memory, completion on `bar`
__device__ __forceinline__ void tma_load_row(uint32_t dst, const CUtensorMap* map, int x4, int y, int f, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(dst),
                 "l"(map), "r"(x4), "r"(y), "r"(f), "r"(bar)
                 : "memory");
}

struct ThrTmaArgs {
    uint8_t* thres;
    uint32_t* bits;
    size_t bits_words;
    int W, H, wpr;
    int idelta;
    int out_mul, out_off;
};

template <int K, int TO, bool U8>
__global__ void __launch_bounds__(TO + 32, 1) k_threshold_tma(const __grid_constant__ CUtensorMap src_map, ThrTmaArgs a) {
    constexpr int R = K / 2, R4 = (R + 3) & ~3, HT = R4 / 4, NV = 4 + 2 * R4, HO = 4 * TO, TW = 2 * HO, CSW = HO + 2 * R4, K2 = K * K;
    constexpr uint32_t BUF_BYTES = CSW * 4;
    constexpr int NT = TO + 2 * HT;            // working threads
    constexpr int GR = 2 * K;                  // rows per group = one unrolled body
    constexpr int NG = THT_NG;                 // groups in flight
    constexpr int ROWB = TW + 32;              // staged bytes per row: columns X0-16 .. X0+TW+15 (TMA: 16-byte aligned start)
    constexpr int ROWP = (ROWB + 127) & ~127;  // row pitch in shared memory: TMA destinations are 128-byte aligned
    constexpr int RH = (THT_RH / GR) * GR;     // output rows per CTA
    constexpr bool OWN = R4 == 4;  // a thread's own column sums stay in registers (two 16-byte shared loads per row instead of three)
    static_assert(NG >= 2 && 2 * R <= GR, "the priming rows borrow the last group slot");
    static_assert(ROWB % 16 == 0 && R4 <= 8, "TMA box: inner extent must be a multiple of 16 bytes");
    // dynamic shared memory: staged rows (NG groups) | 4 column-sum rows (two buffers of two) | barriers (NG groups, priming).
    // The 2R priming rows borrow the last group slot; its group is issued after they are consumed.
    extern __shared__ __align__(128) uint8_t tht_smem[];
    constexpr int PRIME_ROW0 = (NG - 1) * GR;
    constexpr int STAGE_BYTES = NG * GR * ROWP;
    uint8_t* stage = tht_smem;
    uint32_t* cs = reinterpret_cast<uint32_t*>(tht_smem + STAGE_BYTES);
    uint64_t* bars = reinterpret_cast<uint64_t*>(tht_smem + STAGE_BYTES + 4 * BUF_BYTES);
    const int t = threadIdx.x;
    const int X0 = blockIdx.x * TW, y0 = blockIdx.y * RH, f = blockIdx.z;
    const int nout = min(RH, a.H - y0);
    const int ngroups = (nout + GR - 1) / GR;
    const uint32_t s_stage = (uint32_t)__cvta_generic_to_shared(stage);
    const uint32_t s_bars = (uint32_t)__cvta_generic_to_shared(&bars[0]);
    // group g (output rows y0 + g GR ..) needs source rows y0 + R + g GR .. + GR - 1; rows outside the image = nearest row
    auto issue_group = [&](int g) {
        const uint32_t bar = s_bars + 8u * (uint32_t)(g % NG);
        mbar_expect_tx(bar, GR * ROWB);
        const uint32_t dst = s_stage + (uint32_t)((g % NG) * GR * ROWP);
        const int ys = y0 + R + g * GR;
#pragma unroll 1
        for (int r = 0; r < GR; r++) tma_load_row(dst + r * ROWP, &src_map, (X0 - 16) >> 2, min(max(ys + r, 0), a.H - 1), f, bar);
    };
    if (t == 0) {
#pragma unroll
        for (int i = 0; i <= NG; i++) mbar_init(s_bars + 8u * i, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        // priming rows y0-R .. y0+R-1, then the first groups
        const uint32_t pbar = s_bars + 8u * NG;
        mbar_expect_tx(pbar, 2 * R * ROWB);
        for (int r = 0; r < 2 * R; r++)
            tma_load_row(s_stage + (uint32_t)((PRIME_ROW0 + r) * ROWP), &src_map, (X0 - 16) >> 2, min(max(y0 - R + r, 0), a.H - 1), f, pbar);
        for (int g = 0; g < NG - 1 && g < ngroups; g++) issue_group(g);
    }
    __syncthreads();  // barrier words initialised before anybody polls them
    const bool is_out = t < TO;
    // TO need not be a multiple of 32: the last warp with output threads may also hold the halo threads, which do not
    // take part in the shuffles of emit_row
    const unsigned out_mask = __ballot_sync(0xFFFFFFFFu, is_out);
    if (t >= NT) return;  // spare lanes of the halo warp
    // ci: index into a row of cs.  cs[ci] = (V[X0 - R4 + ci], V[X0 + HO - R4 + ci])
    const int ci = is_out ? R4 + 4 * t : (t < TO + HT ? 4 * (t - TO) : R4 + HO + 4 * (t - TO - HT));
    const int ca = X0 - R4 + ci, cb = ca + HO;
    // replicated left/right border: read the nearest in-image word and let the packing PRMT pick byte 0 (left) or 3 (right)
    uint32_t sel[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const uint32_t ja = ca < 0 ? 0u : (ca >= a.W ? 3u : (uint32_t)j), jb = 4u + (cb >= a.W ? 3u : (uint32_t)j);
        sel[j] = ja | (ja << 4) | (jb << 8) | (jb << 12);
    }
    // byte offsets of the thread's two source words inside a staged row (column c sits at byte c - X0 + 16)
    const uint32_t offA = (uint32_t)(min(max(ca, 0), a.W - 4) - X0 + 16), offB = (uint32_t)(min(cb, a.W - 4) - X0 + 16);
    const size_t fo = (size_t)f * a.out_mul + a.out_off;
    uint8_t* orow = a.thres + fo * a.W * a.H + (size_t)y0 * a.W + ca;
    uint32_t* brow = a.bits + fo * a.bits_words + bit_word_index(a.wpr, BIT_PAD + (X0 >> 5) + (t >> 3), y0);
    int btr = (y0 + 1) & 31;  // row inside the bit tile
    const int bjump = a.wpr * BIT_TILE - (BIT_TILE - 1);
    const bool word_t = is_out && (t & 7) == 0;
    const int cst = K2 * a.idelta - (K2 - 1) / 2;  // S >= K2*src + cst  <=>  src - mean <= -idelta
    const uint32_t GC = (uint32_t)((0x8000 - cst) & 0xFFFF) * 0x00010001u;
    const uint32_t M = 0x00FF00FFu;
    const uint32_t s_base = (uint32_t)__cvta_generic_to_shared(cs);
    const uint32_t s_wr = s_base + 4u * ci, s_rd = s_base + 4u * (ci - R4);
    const int nib_shift = 4 * (t & 3);
    uint32_t boff = 0;

    uint32_t ring[K][4];
    uint32_t V0 = 0u, V1 = 0u, V2 = 0u, V3 = 0u;
    // one ring step: the packed row at shared address `row` enters `slot`, the row K steps older leaves the vertical sums
    auto accumulate = [&](uint32_t row, uint32_t* slot, bool first) {
        uint32_t pa, pb;
        asm volatile("ld.shared.b32 %0, [%1];" : "=r"(pa) : "r"(row + offA) : "memory");
        asm volatile("ld.shared.b32 %0, [%1];" : "=r"(pb) : "r"(row + offB) : "memory");
        const uint32_t P0 = prmt_r(pa, pb, sel[0]) & M, P1 = prmt_r(pa, pb, sel[1]) & M, P2 = prmt_r(pa, pb, sel[2]) & M,
                       P3 = prmt_r(pa, pb, sel[3]) & M;
        if (first) {
            V0 += P0, V1 += P1, V2 += P2, V3 += P3;
        } else {
            V0 = V0 + P0 - slot[0];
            V1 = V1 + P1 - slot[1];
            V2 = V2 + P2 - slot[2];
            V3 = V3 + P3 - slot[3];
        }
        slot[0] = P0;
        slot[1] = P1;
        slot[2] = P2;
        slot[3] = P3;
    };
    mbar_wait(s_bars + 8u * NG, 0);
#pragma unroll
    for (int j = 0; j < 2 * R; j++) accumulate(s_stage + (uint32_t)((PRIME_ROW0 + j) * ROWP), ring[j], true);
    __syncthreads();  // the borrowed slot is free again
    if (t == 0 && NG - 1 < ngroups) issue_group(NG - 1);
#pragma unroll
    for (int j = 2 * R; j < K; j++) ring[j][0] = ring[j][1] = ring[j][2] = ring[j][3] = 0u;
    // horizontal window sums, comparison and stores of one output row whose column sums sit at shared offset `rd`
    auto emit_row = [&](uint32_t rd, const uint32_t* c, bool row_ok, const uint32_t* own) {
        uint32_t w[NV];
        if (OWN) {  // the middle four entries are this thread's own sums
            lds128(rd, w[0], w[1], w[2], w[3]);
            lds128(rd + 32u, w[8], w[9], w[10], w[11]);
            w[4] = own[0], w[5] = own[1], w[6] = own[2], w[7] = own[3];
        } else {
#pragma unroll
            for (int q = 0; q < NV / 4; q++) lds128(rd + 16u * q, w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
        }
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
        if (U8 && row_ok) {
            *reinterpret_cast<uint32_t*>(orow) = out_a;
            *reinterpret_cast<uint32_t*>(orow + HO) = out_b;
        }
        const uint32_t nib_a = ((out_a & 0x08040201u) * 0x01010101u) >> 24;
        const uint32_t nib_b = ((out_b & 0x08040201u) * 0x01010101u) >> 24;
        // 8 threads make one 32-bit word per half: two levels carry both halves in one register
        uint32_t x = (nib_a | (nib_b << 16)) << nib_shift;
        x |= __shfl_xor_sync(out_mask, x, 1);
        x |= __shfl_xor_sync(out_mask, x, 2);
        const uint32_t y = __shfl_xor_sync(out_mask, x, 4);
        if (word_t && row_ok) {
            brow[0] = prmt<0x5410>(x, y);
            brow[(HO / 32) * BIT_TILE] = prmt<0x7632>(x, y);
        }
        if (U8) orow += a.W;
        brow += btr == 31 ? bjump : 1;
        btr = (btr + 1) & 31;
    };
    // one group = 2K rows, two rows per CTA barrier (see k_threshold_pair); TAIL: the partial last group of the image
    auto body = [&](uint32_t gbase, int o, auto tail) {
        constexpr bool TAIL = decltype(tail)::value;
#pragma unroll
        for (int jj = 0; jj < GR; jj += 2) {
            uint32_t own[4] = {0u, 0u, 0u, 0u};
#pragma unroll
            for (int q = 0; q < 2; q++) {
                accumulate(gbase + (uint32_t)((jj + q) * ROWP), ring[(2 * R + jj + q) % K], false);
                sts128(s_wr + boff + q * BUF_BYTES, V0, V1, V2, V3);
                if (OWN && q == 0) own[0] = V0, own[1] = V1, own[2] = V2, own[3] = V3;
            }
            __syncthreads();
            if (is_out) {
                const uint32_t cur[4] = {V0, V1, V2, V3};
#pragma unroll
                for (int q = 0; q < 2; q++)
                    emit_row(s_rd + boff + q * BUF_BYTES, ring[(R + jj + q) % K], !TAIL || o + jj + q < nout, q == 0 ? own : cur);
            }
            boff = 2 * BUF_BYTES - boff;
        }
    };
    for (int g = 0; g < ngroups; g++) {
        const int slot = g % NG;
        mbar_wait(s_bars + 8u * (uint32_t)slot, (uint32_t)((g / NG) & 1));
        const uint32_t gbase = s_stage + (uint32_t)(slot * GR * ROWP);
        if ((g + 1) * GR <= nout) body(gbase, g * GR, std::false_type{});
        else body(gbase, g * GR, std::true_type{});
        // every thread is past its last read of this slot (the body ends behind a CTA barrier): refill it
        if (t == 0 && g + NG < ngroups) issue_group(g + NG);
    }
}

// ---- block sizes 13 .. 21 ---------------------------------------------------------------------------------------
// The window sums of K >= 13 do not fit the 16-bit lanes (K^2 * 255 >= 2^15) and a register ring of K packed rows per
// column pair does not fit the register file, so the round-1 fallback k_threshold_fast<K> spent 27 instructions per pixel
// (it was 40 % of config C5, ADPT 21/7).  Same TMA staging as above with three changes:
//   * no register ring: the staged tile keeps the last K + 2 GR + 3 source rows, and the row that leaves the vertical window
//     (and the centre row of the mean test) is read from it again and unpacked;
//   * the vertical sums stay lane-paired 16-bit (K * 255 < 2^13); the horizontal window is added in packed chunks that
//     cannot overflow (floor(65535 / (255 K)) terms) and continued in two 32-bit accumulators per pixel pair;
//   * the mean test is a 32-bit comparison per pixel: S - cst - K^2 * src >= 0.
template <int K, int TO, bool U8>
__global__ void __launch_bounds__(TO + 32, 1) k_threshold_tma_wide(const __grid_constant__ CUtensorMap src_map, ThrTmaArgs a) {
    constexpr int R = K / 2, R4 = (R + 3) & ~3, HT = R4 / 4, NV = 4 + 2 * R4, HO = 4 * TO, TW = 2 * HO, CSW = HO + 2 * R4, K2 = K * K;
    constexpr uint32_t BUF_BYTES = CSW * 4;
    constexpr int NT = TO + 2 * HT;
    constexpr int GR = THW_GR;                 // rows per TMA group = one unrolled body
    constexpr int NS = K + 2 * GR + 3;         // staged rows (ring); row NS is a row of zeros
    constexpr int ROWB = TW + 32, ROWP = (ROWB + 127) & ~127;
    constexpr int RH = (THT_RH / GR) * GR;
    constexpr int CH = 65535 / (255 * K);      // packed terms that cannot overflow a 16-bit lane
    static_assert(R4 <= 16, "halo of the staged tile is 16 columns");
    extern __shared__ __align__(128) uint8_t tht_smem[];
    constexpr int STAGE_BYTES = (NS + 1) * ROWP;
    uint8_t* stage = tht_smem;
    uint32_t* cs = reinterpret_cast<uint32_t*>(tht_smem + STAGE_BYTES);
    uint64_t* bars = reinterpret_cast<uint64_t*>(tht_smem + STAGE_BYTES + 4 * BUF_BYTES);  // 3 group slots + priming
    const int t = threadIdx.x;
    const int X0 = blockIdx.x * TW, y0 = blockIdx.y * RH, f = blockIdx.z;
    const int nout = min(RH, a.H - y0);
    const int ngroups = (nout + GR - 1) / GR;
    const uint32_t s_stage = (uint32_t)__cvta_generic_to_shared(stage);
    const uint32_t s_bars = (uint32_t)__cvta_generic_to_shared(&bars[0]);
    // stream row s = image row y0 - R + s (clamped: replicated border) lives in ring slot s % NS
    auto issue_rows = [&](int s0, int n, uint32_t bar) {
        mbar_expect_tx(bar, (uint32_t)(n * ROWB));
#pragma unroll 1
        for (int r = 0; r < n; r++) {
            const int srow = s0 + r;
            tma_load_row(s_stage + (uint32_t)((srow % NS) * ROWP), &src_map, (X0 - 16) >> 2, min(max(y0 - R + srow, 0), a.H - 1), f, bar);
        }
    };
    for (int i = 4 * t; i < ROWP; i += 4 * (int)blockDim.x) *reinterpret_cast<uint32_t*>(stage + (size_t)NS * ROWP + i) = 0u;
    if (t == 0) {
#pragma unroll
        for (int i = 0; i < 4; i++) mbar_init(s_bars + 8u * i, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        issue_rows(0, 2 * R, s_bars + 8u * 3);  // priming rows
        for (int g = 0; g < 2 && g < ngroups; g++) issue_rows(2 * R + g * GR, GR, s_bars + 8u * (uint32_t)g);
    }
    __syncthreads();
    const bool is_out = t < TO;
    const unsigned out_mask = __ballot_sync(0xFFFFFFFFu, is_out);
    if (t >= NT) return;
    const int ci = is_out ? R4 + 4 * t : (t < TO + HT ? 4 * (t - TO) : R4 + HO + 4 * (t - TO - HT));
    const int ca = X0 - R4 + ci, cb = ca + HO;
    uint32_t sel[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const uint32_t ja = ca < 0 ? 0u : (ca >= a.W ? 3u : (uint32_t)j), jb = 4u + (cb >= a.W ? 3u : (uint32_t)j);
        sel[j] = ja | (ja << 4) | (jb << 8) | (jb << 12);
    }
    const uint32_t offA = s_stage + (uint32_t)(min(max(ca, 0), a.W - 4) - X0 + 16), offB = s_stage + (uint32_t)(min(cb, a.W - 4) - X0 + 16);
    const size_t fo = (size_t)f * a.out_mul + a.out_off;
    uint8_t* orow = a.thres + fo * a.W * a.H + (size_t)y0 * a.W + ca;
    uint32_t* brow = a.bits + fo * a.bits_words + bit_word_index(a.wpr, BIT_PAD + (X0 >> 5) + (t >> 3), y0);
    int btr = (y0 + 1) & 31;
    const int bjump = a.wpr * BIT_TILE - (BIT_TILE - 1);
    const bool word_t = is_out && (t & 7) == 0;
    const int cst = K2 * a.idelta - (K2 - 1) / 2;  // S >= K2*src + cst  <=>  src - mean <= -idelta
    const uint32_t M = 0x00FF00FFu;
    const uint32_t s_base = (uint32_t)__cvta_generic_to_shared(cs);
    const uint32_t s_wr = s_base + 4u * ci, s_rd = s_base + 4u * (ci - R4);
    const int nib_shift = 4 * (t & 3);
    uint32_t boff = 0;
    uint32_t V0 = 0u, V1 = 0u, V2 = 0u, V3 = 0u;
    // the four packed pixel pairs of this thread in the staged row at byte offset `row`
    auto unpack = [&](uint32_t row, uint32_t* P) {
        uint32_t pa, pb;
        asm volatile("ld.shared.b32 %0, [%1];" : "=r"(pa) : "r"(offA + row) : "memory");
        asm volatile("ld.shared.b32 %0, [%1];" : "=r"(pb) : "r"(offB + row) : "memory");
#pragma unroll
        for (int j = 0; j < 4; j++) P[j] = prmt_r(pa, pb, sel[j]) & M;
    };
    constexpr uint32_t RING_BYTES = (uint32_t)NS * ROWP;
    auto adv = [&](uint32_t& off) { off = off + ROWP >= RING_BYTES ? 0u : off + ROWP; };
    mbar_wait(s_bars + 8u * 3, 0);
#pragma unroll 4
    for (int srow = 0; srow < 2 * R; srow++) {
        uint32_t P[4];
        unpack((uint32_t)(srow * ROWP), P);
        V0 += P[0], V1 += P[1], V2 += P[2], V3 += P[3];
    }
    uint32_t off_new = (uint32_t)(2 * R * ROWP), off_old = RING_BYTES /* the zero row: nothing leaves the window yet */,
             off_c = (uint32_t)(R * ROWP);
    auto accumulate = [&]() {
        uint32_t P[4], Q[4];
        unpack(off_new, P);
        unpack(off_old, Q);
        V0 = V0 + P[0] - Q[0];
        V1 = V1 + P[1] - Q[1];
        V2 = V2 + P[2] - Q[2];
        V3 = V3 + P[3] - Q[3];
        adv(off_new);
        adv(off_old);  // from the zero row (offset RING_BYTES) this wraps to slot 0 = stream row 0
    };
    auto emit_row = [&](uint32_t rd, bool row_ok, const uint32_t* own) {
        uint32_t c[4];
        unpack(off_c, c);
        adv(off_c);
        uint32_t w[NV];
#pragma unroll
        for (int q = 0; q < R4 / 4; q++) {
            lds128(rd + 16u * q, w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
            lds128(rd + 16u * (R4 / 4 + 1 + q), w[R4 + 4 + 4 * q], w[R4 + 5 + 4 * q], w[R4 + 6 + 4 * q], w[R4 + 7 + 4 * q]);
        }
        w[R4] = own[0], w[R4 + 1] = own[1], w[R4 + 2] = own[2], w[R4 + 3] = own[3];
        // window of pixel 0: packed chunk sums, widened to one 32-bit accumulator per half
        int32_t Sa = -cst, Sb = -cst;
#pragma unroll
        for (int c0 = 0; c0 < K; c0 += CH) {
            uint32_t g = 0u;
#pragma unroll
            for (int d = c0; d < c0 + CH && d < K; d++) g += w[R4 - R + d];
            Sa += (int32_t)(g & 0xFFFFu);
            Sb += (int32_t)(g >> 16);
        }
        uint32_t nib_a = 0u, nib_b = 0u;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            if (j > 0) {  // slide the window one column
                const uint32_t wo = w[R4 - R + j - 1], wi = w[R4 + R + j];
                Sa += (int32_t)(wi & 0xFFFFu) - (int32_t)(wo & 0xFFFFu);
                Sb += (int32_t)(wi >> 16) - (int32_t)(wo >> 16);
            }
            const int32_t Da = Sa - K2 * (int32_t)(c[j] & 0xFFFFu), Db = Sb - K2 * (int32_t)(c[j] >> 16);
            nib_a |= ((uint32_t)~Da >> 31) << j;  // foreground <=> D >= 0
            nib_b |= ((uint32_t)~Db >> 31) << j;
        }
        if (U8 && row_ok) {
            *reinterpret_cast<uint32_t*>(orow) = bits4_to_bytes(nib_a);
            *reinterpret_cast<uint32_t*>(orow + HO) = bits4_to_bytes(nib_b);
        }
        uint32_t x = (nib_a | (nib_b << 16)) << nib_shift;
        x |= __shfl_xor_sync(out_mask, x, 1);
        x |= __shfl_xor_sync(out_mask, x, 2);
        const uint32_t y = __shfl_xor_sync(out_mask, x, 4);
        if (word_t && row_ok) {
            brow[0] = prmt<0x5410>(x, y);
            brow[(HO / 32) * BIT_TILE] = prmt<0x7632>(x, y);
        }
        if (U8) orow += a.W;
        brow += btr == 31 ? bjump : 1;
        btr = (btr + 1) & 31;
    };
    int o = 0;
    for (int g = 0; g < ngroups; g++) {
        mbar_wait(s_bars + 8u * (uint32_t)(g % 3), (uint32_t)((g / 3) & 1));
#pragma unroll
        for (int jj = 0; jj < GR; jj += 2) {
            accumulate();
            sts128(s_wr + boff, V0, V1, V2, V3);
            const uint32_t own_a[4] = {V0, V1, V2, V3};
            accumulate();
            sts128(s_wr + boff + BUF_BYTES, V0, V1, V2, V3);
            __syncthreads();
            if (is_out) {
                const uint32_t own_b[4] = {V0, V1, V2, V3};
                emit_row(s_rd + boff, o < nout, own_a);
                emit_row(s_rd + boff + BUF_BYTES, o + 1 < nout, own_b);
            }
            o += 2;
            boff = 2 * BUF_BYTES - boff;
        }
        // group g+2 overwrites stream rows <= GR g + GR - 5; the centre rows still being read are >= R + GR g + GR - 2
        if (t == 0 && g + 2 < ngroups) issue_rows(2 * R + (g + 2) * GR, GR, s_bars + 8u * (uint32_t)((g + 2) % 3));
    }
}

// ---- host side ---------------------------------------------------------------------------------------------------
typedef CUresult (*ab_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                       const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                       CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline ab_encode_tiled_fn tensor_map_encoder() {
    static ab_encode_tiled_fn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) p = nullptr;
        return (ab_encode_tiled_fn)p;
    }();
    return fn;
}

// the TO whose tile width 8*TO divides W (widest first); 0 if none
inline int threshold_tma_tile(int W) {
    for (int to : {96, 120, 80, 64, 40})  // (8 TO + 32) / 4 <= 256: the TMA box limit
        if (W % (8 * to) == 0) return to;
    return 0;
}

constexpr size_t threshold_tma_wide_smem(int K, int TO) {
    const int R = K / 2, R4 = (R + 3) & ~3, HO = 4 * TO, TW = 2 * HO, CSW = HO + 2 * R4;
    return (size_t)(K + 2 * THW_GR + 4) * (size_t)((TW + 32 + 127) & ~127) + 4 * (size_t)CSW * 4 + 8 * 4;
}
constexpr size_t threshold_tma_smem(int K, int TO) {
    const int R = K / 2, R4 = (R + 3) & ~3, HO = 4 * TO, TW = 2 * HO, CSW = HO + 2 * R4;
    return (size_t)(THT_NG * 2 * K) * (size_t)((TW + 32 + 127) & ~127) + 4 * (size_t)CSW * 4 + 8 * (THT_NG + 1);
}
template <class KERNEL>
inline void threshold_tma_launch(KERNEL kern, dim3 grid, int threads, size_t smem, cudaStream_t st, const CUtensorMap& map, const ThrTmaArgs& ta) {
    // more than 48 KB of dynamic shared memory must be allowed once per kernel (all instantiations share this function's type,
    // so the kernels already raised are remembered by address)
    static const void* raised[64];
    static int n_raised = 0;
    if (smem > 48 * 1024) {
        bool seen = false;
        for (int i = 0; i < n_raised; i++) seen |= raised[i] == (const void*)kern;
        if (!seen) {
            cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (n_raised < 64) raised[n_raised++] = (const void*)kern;
        }
    }
    kern<<<grid, threads, smem, st>>>(map, ta);
}

// returns false when the TMA path does not apply (alignment, tile divisibility, lane budget): the caller falls back
inline bool launch_threshold_tma(const ThrArgs& a, int B, cudaStream_t st) {
    const int K2 = a.k * a.k;
    const long long cst = (long long)K2 * a.idelta - (K2 - 1) / 2;
    if (a.k < 3 || a.k > 21 || !(a.k & 1) || (a.W & 3)) return false;
    const bool wide = a.k >= 13 || K2 * 255LL + (cst < 0 ? -cst : cst) >= 0x8000;  // the window sums leave the 16-bit lanes
    if (wide && a.k < 13) return false;
    if ((((uintptr_t)a.grey) | a.grey_row | a.grey_frame) & 15) return false;  // TMA: 16-byte aligned base and strides
    const int to = threshold_tma_tile(a.W);
    ab_encode_tiled_fn enc = tensor_map_encoder();
    if (!to || !enc) return false;
    const int tw = 8 * to;
    CUtensorMap map;
    const cuuint64_t gdim[3] = {(cuuint64_t)(a.W / 4), (cuuint64_t)a.H, (cuuint64_t)B};
    const cuuint64_t gstr[2] = {(cuuint64_t)a.grey_row, (cuuint64_t)a.grey_frame};
    const cuuint32_t box[3] = {(cuuint32_t)((tw + 32) / 4), 1u, 1u}, estr[3] = {1u, 1u, 1u};
    if (enc(&map, CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, (void*)a.grey, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
        return false;
    ThrTmaArgs ta{a.thres, a.bits, a.bits_words, a.W, a.H, a.wpr, a.idelta, a.out_mul, a.out_off};
    const int rh = wide ? (THT_RH / THW_GR) * THW_GR : (THT_RH / (2 * a.k)) * (2 * a.k);
    dim3 grid(a.W / tw, (a.H + rh - 1) / rh, B);
    if (wide) {
#define AB_THW_TO(KK, TT)                                                                                                \
    if (to == TT) {                                                                                                      \
        const size_t smem = threshold_tma_wide_smem(KK, TT);                                                             \
        if (a.skip_u8) threshold_tma_launch(k_threshold_tma_wide<KK, TT, false>, grid, TT + 32, smem, st, map, ta);      \
        else threshold_tma_launch(k_threshold_tma_wide<KK, TT, true>, grid, TT + 32, smem, st, map, ta);                 \
        return true;                                                                                                     \
    }
#define AB_THW_CASE(KK) \
    case KK:            \
        AB_THW_TO(KK, 96) AB_THW_TO(KK, 120) AB_THW_TO(KK, 80) AB_THW_TO(KK, 40) return false;
        switch (a.k) {
            AB_THW_CASE(13)
            AB_THW_CASE(15)
            AB_THW_CASE(17)
            AB_THW_CASE(19)
            AB_THW_CASE(21)
            default:
                return false;
        }
#undef AB_THW_CASE
#undef AB_THW_TO
    }
#define AB_THT_TO(KK, TT)                                                                        \
    if (to == TT) {                                                                              \
        const size_t smem = threshold_tma_smem(KK, TT);                                          \
        if (a.skip_u8) threshold_tma_launch(k_threshold_tma<KK, TT, false>, grid, TT + 32, smem, st, map, ta); \
        else threshold_tma_launch(k_threshold_tma<KK, TT, true>, grid, TT + 32, smem, st, map, ta);            \
        return true;                                                                             \
    }
#define AB_THT_CASE(KK) \
    case KK:            \
        AB_THT_TO(KK, 96) AB_THT_TO(KK, 120) AB_THT_TO(KK, 80) AB_THT_TO(KK, 64) AB_THT_TO(KK, 40) return false;
    switch (a.k) {
        AB_THT_CASE(3)
        AB_THT_CASE(5)
        AB_THT_CASE(7)
        AB_THT_CASE(9)
        AB_THT_CASE(11)
        default:
            return false;
    }
#undef AB_THT_CASE
#undef AB_THT_TO
}

}  // namespace ab
