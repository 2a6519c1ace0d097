// Stage 3: per-candidate identification (src/markerdetector.cpp:350-356), four kernels:
//   k_homography (thread / candidate)  getPerspectiveTransform + inverse            (MarkerDetector::warp, :684-697)
//   k_sample     (warp / candidate)    warpPerspective(INTER_NEAREST) -> canonical image + 256-bin histogram
//   k_otsu       (thread / candidate)  cv::threshold(BINARY|OTSU) threshold search
//   k_identify   (warp / candidate)    majority vote per cell, FiducidalMarkers::detect (src/arucofidmarkers.cpp:438-452)
//                                      or HighlyReliableMarkers::detect (src/highlyreliablemarkers.cpp:332-383)
// The serial f64 chains (8x8 LU, the Otsu recurrence -- both must follow OpenCV's operation order to stay bit-exact)
// get a lane each instead of a warp each; the pixel-parallel parts get a warp per candidate.
#pragma once
#include "ab_device.cuh"

namespace ab {

constexpr int MAX_WARP_SIZE = 128;  // S <= 128
constexpr int MAX_CELLS = 100;      // (n+2)^2 with n <= 8
constexpr int DECODE_WARPS = 4;
constexpr int DECODE_LIST = 1024;   // per-warp list of pixels that need the exact f64 coordinate

__device__ __forceinline__ int hrm_decode(const HrmDict& D, const uint8_t* cells, int ncell, int* nrot, int lane) {
    // cells: (n+2)^2 majority bits; HRM ignores the border cells (highlyreliablemarkers.cpp:345)
    const int n = D.n;
    uint8_t code[64];
    for (int y = 0; y < n; y++)
        for (int x = 0; x < n; x++) code[y * n + x] = cells[(y + 1) * ncell + x + 1];
    uint64_t bits[4];
    uint32_t ids[4];
    hrm_rotations(code, n, bits, ids);
    // 1. exact lookup of the four folded ids in the balanced tree (findId, :483-496)
    for (int r = 0; r < 4; r++) {
        int pos = D.root;
        while (pos != -1) {
            uint32_t pid = D.ord_ids[pos];
            if (pid == ids[r]) {
                *nrot = r;
                return D.ord_pos[pos];
            }
            pos = pid < ids[r] ? D.tree[2 * pos + 1] : D.tree[2 * pos];
        }
    }
    // 2. error correction: min over dictionary of min over rotations (Dictionary::distance, :277-289),
    //    first strict minimum wins in (marker, rotation) order
    unsigned best = 0xFFFFFFFFu;  // (dist << 16) | (marker << 2) | rot
    for (int i = lane; i < D.count; i += 32) {
        uint64_t d0 = D.bits[i];
        unsigned res = (unsigned)(n * n), mr = 0;
        for (unsigned r = 0; r < 4; r++) {
            unsigned hd = (unsigned)__popcll(d0 ^ bits[r]);
            if (hd < res) {
                res = hd;
                mr = r;
            }
        }
        if (res < (unsigned)(n * n)) {
            unsigned key = (res << 16) | ((unsigned)i << 2) | mr;
            best = min(best, key);
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) best = min(best, __shfl_xor_sync(0xFFFFFFFFu, best, d));
    if (best != 0xFFFFFFFFu && (int)(best >> 16) <= D.correction) {
        *nrot = (int)(best & 3u);
        return (int)((best >> 2) & 0x3FFFu);
    }
    *nrot = 0;
    return -1;
}

// ---------------------------------------------------------------------------------------------------
// 1. k_homography: one THREAD per candidate.  getPerspectiveTransform's 8x8 LU and the 3x3 inverse are serial
//    f64 chains that must follow OpenCV's operation order; one per lane keeps 32 of them busy per warp (ncu r1k:
//    as a lane-0 prologue of the warp-per-candidate kernel they were 16 % of its stall samples).
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(64) k_homography(Batch b) {
    const int f = blockIdx.y, ci = blockIdx.x * blockDim.x + threadIdx.x;
    if (ci >= (int)b.n_cands[f] || ci >= b.cap_c) return;
    const int S = b.S;
    const CandRec* cand = b.cands + (size_t)f * b.cap_c + ci;
    CandAux* ax = b.aux + (size_t)f * b.cap_c + ci;
    float src[8];
    for (int i = 0; i < 8; i++) src[i] = cand->c[i];
    const float dst[8] = {0.f, 0.f, (float)(S - 1), 0.f, (float)(S - 1), (float)(S - 1), 0.f, (float)(S - 1)};
    double M[9], Mi[9];
    const bool ok = perspective_transform(src, dst, M) && invert3(M, Mi);
    for (int i = 0; i < 9; i++) ax->Mi[i] = ok ? Mi[i] : 0.0;
    ax->ok = ok;
    ax->thr = 0;
}

// ---------------------------------------------------------------------------------------------------
// 2. k_sample: one WARP per candidate: warpPerspective(INTER_NEAREST) into the canonical image (global; getCandidates,
//    host-callback decoders and k_identify read it) and its 256-bin histogram.
//    Filtered arithmetic: OpenCV's source coordinate is rint() of an f64 expression.  An f32 evaluation (error
//    << 0.05 px for |coord| < 32768) decides every pixel whose coordinate is not within its error bound of a rounding
//    boundary -- the integer it rounds to is then provably the same; the rest (a few % on tilted markers) is collected
//    by ballot compaction and redone densely with the exact f64 sequence.  A lane owns 4 adjacent destination pixels per
//    step: their 4 gathers are in flight together (r1k: 23 % of the stall samples sat on the single gather) and
//    the canonical image is written as 32-bit words.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32 * DECODE_WARPS) k_sample(Batch b) {
    __shared__ int s_hist_all[DECODE_WARPS][256];
    __shared__ unsigned short s_list_all[DECODE_WARPS][DECODE_LIST];
    const int f = blockIdx.y, lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int ci = blockIdx.x * DECODE_WARPS + wib;
    if (ci >= (int)b.n_cands[f] || ci >= b.cap_c) return;  // whole warp leaves; only warp-level sync below
    const unsigned FULL = 0xFFFFFFFFu;
    const int S = b.S, SS = S * S;
    int* s_hist = s_hist_all[wib];
    unsigned short* s_list = s_list_all[wib];
    const size_t slot = (size_t)f * b.cap_c + ci;
    const CandAux* ax = b.aux + slot;
    const uint8_t* grey = b.grey + (size_t)f * b.grey_frame;
    uint8_t* canon = b.canon + slot * (size_t)SS;
    const int bw = warp_block_width(S);
    const bool ok = ax->ok != 0;
    for (int i = lane; i < 256; i += 32) s_hist[i] = 0;
    __syncwarp();
    if (!ok) {  // degenerate quad: the reference warps nothing useful either; an all-zero image decodes to "no marker"
        for (int i = lane; i < SS; i += 32) canon[i] = 0;
        if (lane == 0) s_hist[0] = SS;
    } else {
        float Mf[9];
#pragma unroll
        for (int q = 0; q < 9; q++) Mf[q] = (float)ax->Mi[q];
        // Forward error bound of the f32 evaluation, once per candidate: |error(fx)| <= u' * (|M0 x| + |M1 y| + |M2|) / |den|
        // with u' covering ~12 roundings (unit roundoff 6e-8; 4e-6 leaves > 5x slack).  The bound is a ratio of affine
        // functions with positive terms, so over the destination square it peaks at a corner -- unless den changes
        // sign inside the square (horizon through the marker), in which case every pixel takes the exact path.
        float gx, gy;  // a coordinate is trusted when it is more than (0.5 - g) away from a rounding boundary
        {
            const float aM0 = fabsf(Mf[0]), aM1 = fabsf(Mf[1]), aM2 = fabsf(Mf[2]), aM3 = fabsf(Mf[3]), aM4 = fabsf(Mf[4]), aM5 = fabsf(Mf[5]);
            const float e = (float)(S - 1);
            float mx = 0.f, my = 0.f;
            int pos = 0, neg = 0;
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const float cx = (c & 1) ? e : 0.f, cy = (c & 2) ? e : 0.f;
                const float den = __fmaf_rn(Mf[6], cx, __fmaf_rn(Mf[7], cy, Mf[8]));
                pos += den > 0.f;
                neg += den < 0.f;
                const float iad = 1.0f / fabsf(den);
                mx = fmaxf(mx, __fmaf_rn(aM0, cx, __fmaf_rn(aM1, cy, aM2)) * iad);
                my = fmaxf(my, __fmaf_rn(aM3, cx, __fmaf_rn(aM4, cy, aM5)) * iad);
            }
            const bool one_sign = pos == 4 || neg == 4;
            gx = one_sign ? 0.5f - (4e-6f * mx + 2e-4f) : -1.f;
            gy = one_sign ? 0.5f - (4e-6f * my + 2e-4f) : -1.f;
        }
        const float invS = 1.0f / (float)S;
        const bool words = (SS & 3) == 0;
        int nunc = 0;
        for (int i0 = 0; i0 < SS; i0 += 128) {
            uint32_t v[4];
            bool unc[4], act[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int i = i0 + 4 * lane + u;
                act[u] = i < SS;
                unc[u] = false;
                v[u] = 0;
                if (act[u]) {
                    const int y = (int)(((float)i + 0.5f) * invS), x = i - y * S;  // exact: the fraction is >= 0.5/S away from an integer
                    const float fxp = (float)x, fyp = (float)y;
                    const float den = __fmaf_rn(Mf[6], fxp, __fmaf_rn(Mf[7], fyp, Mf[8]));
                    float iden;
                    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(iden) : "f"(den));  // <= 1 ulp: inside the bound's slack
                    const float fx = __fmaf_rn(Mf[0], fxp, __fmaf_rn(Mf[1], fyp, Mf[2])) * iden;
                    const float fy = __fmaf_rn(Mf[3], fxp, __fmaf_rn(Mf[4], fyp, Mf[5])) * iden;
                    const float rx = rintf(fx), ry = rintf(fy);
                    unc[u] = !(fabsf(fx) < 32768.f && fabsf(fy) < 32768.f) || !(fabsf(fx - rx) < gx) || !(fabsf(fy - ry) < gy);
                    if (!unc[u]) {
                        const int sx = (int)rx, sy = (int)ry;
                        if (sx >= 0 && sy >= 0 && sx < b.W && sy < b.H) v[u] = grey[(size_t)sy * b.grey_row + sx];
                    }
                }
            }
            if (words) {
                if (act[0]) *reinterpret_cast<uint32_t*>(canon + i0 + 4 * lane) = v[0] | (v[1] << 8) | (v[2] << 16) | (v[3] << 24);
            } else {
#pragma unroll
                for (int u = 0; u < 4; u++)
                    if (act[u] && !unc[u]) canon[i0 + 4 * lane + u] = (uint8_t)v[u];
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
                // histogram: lanes holding the same grey level are matched, one of them adds the group size
                // (shared-memory atomics on a bimodal image serialise almost completely: 18 % of the stall samples in r1e)
                const bool cnt = act[u] && !unc[u];
                const unsigned key = cnt ? v[u] : 0x100u + (unsigned)lane;
                const unsigned peers = __match_any_sync(FULL, key);
                if (cnt && lane == __ffs((int)peers) - 1) s_hist[key] += __popc(peers);
                const unsigned m = __ballot_sync(FULL, unc[u]);
                if (m) {
                    const int pos = nunc + __popc(m & ((1u << lane) - 1u));
                    if (unc[u]) {
                        const int i = i0 + 4 * lane + u;
                        if (pos < DECODE_LIST) {
                            s_list[pos] = (unsigned short)i;
                        } else {  // list full: do it now.  Ordinary quads fill the list: an axis-aligned side of an odd
                                  // multiple of (S-1)/2 puts every other sample row and column on a half pixel and defers
                                  // 3/4 of the S*S pixels, more than DECODE_LIST from S = 37 on
                            const int y = i / S, x = i - y * S;
                            int sx, sy;
                            warp_src_coord(ax->Mi, x, y, bw, &sx, &sy);
                            uint8_t vv = 0;
                            if (sx >= 0 && sy >= 0 && sx < b.W && sy < b.H) vv = grey[(size_t)sy * b.grey_row + sx];
                            canon[i] = vv;
                            atomicAdd(&s_hist[vv], 1);
                        }
                    }
                    nunc += __popc(m);
                }
            }
        }
        __syncwarp();
        const int n2 = min(nunc, DECODE_LIST);
        for (int k = lane; k < n2; k += 32) {
            const int i = (int)s_list[k];
            const int y = i / S, x = i - y * S;
            int sx, sy;
            warp_src_coord(ax->Mi, x, y, bw, &sx, &sy);
            uint8_t vv = 0;
            if (sx >= 0 && sy >= 0 && sx < b.W && sy < b.H) vv = grey[(size_t)sy * b.grey_row + sx];
            canon[i] = vv;
            atomicAdd(&s_hist[vv], 1);
        }
    }
    __syncwarp();
    // histogram -> global as 256 x u16 (S <= 128: counts < 65536 unless the image is constant, which saturates harmlessly
    // below: a constant image has one bin = S*S <= 16384)
    uint32_t w4[4];
#pragma unroll
    for (int q = 0; q < 4; q++) w4[q] = (uint32_t)s_hist[8 * lane + 2 * q] | ((uint32_t)s_hist[8 * lane + 2 * q + 1] << 16);
    reinterpret_cast<uint4*>(b.hist + slot * 256)[lane] = make_uint4(w4[0], w4[1], w4[2], w4[3]);
}

// ---------------------------------------------------------------------------------------------------
// 3. k_otsu: one THREAD per candidate runs cv::threshold(BINARY|OTSU)'s sequential search (otsu_threshold, ab_math.cuh)
//    on its histogram.  The (q1, mu1) recurrence -- an f64 division per bin whose rounding sequence must be
//    reproduced -- was 40 % of the instructions of the warp-per-candidate kernel at 1/32 lane use (ncu r1k).
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) k_otsu(Batch b) {
    __shared__ int s_h[32 * 257];  // row stride 257: lane c walks bank (c + i) % 32
    const int f = blockIdx.y, lane = threadIdx.x, c0 = blockIdx.x * 32;
    const int nc = min((int)b.n_cands[f], b.cap_c);
    if (c0 >= nc) return;
    const int rows = min(32, nc - c0);
    for (int r = 0; r < rows; r++) {
        const uint4 u = reinterpret_cast<const uint4*>(b.hist + ((size_t)f * b.cap_c + c0 + r) * 256)[lane];
        int* d = s_h + r * 257 + 8 * lane;
        d[0] = (int)(u.x & 0xFFFFu);
        d[1] = (int)(u.x >> 16);
        d[2] = (int)(u.y & 0xFFFFu);
        d[3] = (int)(u.y >> 16);
        d[4] = (int)(u.z & 0xFFFFu);
        d[5] = (int)(u.z >> 16);
        d[6] = (int)(u.w & 0xFFFFu);
        d[7] = (int)(u.w >> 16);
    }
    __syncwarp();
    if (lane < rows) b.aux[(size_t)f * b.cap_c + c0 + lane].thr = otsu_threshold(s_h + lane * 257, b.S * b.S);
}

inline size_t identify_smem_per_warp(int S) { return (((size_t)S * S + 15) & ~(size_t)15) + 112; }

// ---------------------------------------------------------------------------------------------------
// 4. k_identify: one WARP per candidate: majority vote per cell of the Otsu-binarised canonical image, then
//    FiducidalMarkers::detect (src/arucofidmarkers.cpp:438-452) or HighlyReliableMarkers::detect
//    (src/highlyreliablemarkers.cpp:332-383).  grid = (ceil(cap_c / DECODE_WARPS), B)
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32 * DECODE_WARPS) k_identify(Batch b) {
    extern __shared__ __align__(16) unsigned char s_raw[];
    const int f = blockIdx.y, lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int ci = blockIdx.x * DECODE_WARPS + wib;
    if (ci >= (int)b.n_cands[f] || ci >= b.cap_c) return;
    const int S = b.S, SS = S * S;
    const size_t img_bytes = ((size_t)SS + 15) & ~(size_t)15;
    unsigned char* base = s_raw + (size_t)wib * (img_bytes + 112);
    uint8_t* s_img = base;
    uint8_t* s_cells = base + img_bytes;
    const size_t slot = (size_t)f * b.cap_c + ci;
    CandRec* cand = b.cands + slot;
    const uint8_t* canon = b.canon + slot * (size_t)SS;
    const int thr = b.aux[slot].thr;
    if ((SS & 3) == 0) {
        for (int i = lane; i < SS / 4; i += 32) reinterpret_cast<uint32_t*>(s_img)[i] = reinterpret_cast<const uint32_t*>(canon)[i];
    } else {
        for (int i = lane; i < SS; i += 32) s_img[i] = canon[i];
    }
    __syncwarp();
    const int ncell = (b.decoder == AB_DECODER_HRM) ? b.dict.n + 2 : 7;
    const int cell = S / ncell;
    for (int cidx = lane; cidx < ncell * ncell; cidx += 32) {  // one lane per cell: no atomics
        const int cy = cidx / ncell, cx = cidx - cy * ncell;
        int cnt = 0;
        for (int yy = 0; yy < cell; yy++) {
            const uint8_t* rowp = s_img + (cy * cell + yy) * S + cx * cell;
            for (int xx = 0; xx < cell; xx++) cnt += rowp[xx] > thr;
        }
        s_cells[cidx] = cnt > (cell * cell) / 2;
    }
    __syncwarp();
    if (b.decoder == AB_DECODER_HRM) {
        int nrot = 0;
        int id = hrm_decode(b.dict, s_cells, ncell, &nrot, lane);
        if (lane == 0) {
            cand->id = id;
            cand->nrot = nrot;
        }
    } else if (lane == 0) {
        int nrot = 0;
        int id = fid_decode(s_cells, &nrot);
        cand->id = id;
        cand->nrot = nrot;
    }
}

// public worker MarkerDetector::warp for one quad (grid 1)
__global__ void k_warp_single(const uint8_t* grey, int W, int H, size_t row, const float* quad, int S, uint8_t* out) {
    __shared__ double s_Mi[9];
    __shared__ int s_ok;
    if (threadIdx.x == 0) {
        float dst[8] = {0.f, 0.f, (float)(S - 1), 0.f, (float)(S - 1), (float)(S - 1), 0.f, (float)(S - 1)};
        float q[8];
        for (int i = 0; i < 8; i++) q[i] = quad[i];
        double M[9], Mi[9];
        bool ok = perspective_transform(q, dst, M) && invert3(M, Mi);
        s_ok = ok;
        if (ok)
            for (int i = 0; i < 9; i++) s_Mi[i] = Mi[i];
    }
    __syncthreads();
    const int bw = warp_block_width(S);
    for (int i = threadIdx.x; i < S * S; i += blockDim.x) {
        int y = i / S, x = i - y * S;
        uint8_t v = 0;
        if (s_ok) {
            int sx, sy;
            warp_src_coord(s_Mi, x, y, bw, &sx, &sy);
            if (sx >= 0 && sy >= 0 && sx < W && sy < H) v = grey[(size_t)sy * row + sx];
        }
        out[i] = v;
    }
}

}  // namespace ab
