// Stage 5: result assembly (src/markerdetector.cpp:364-382, 416-467).
//   k_finalize: one CTA per frame -- corner rotation by nRotations, stable sort by id, duplicate-id removal (keep the
//               larger perimeter), border filter; writes the marker list without poses.
//   k_pose:     one thread per surviving marker, one WARP per CTA -- planar PnP (cv::solvePnP ITERATIVE) in f64.  The LM
//               chain of a marker is ~20 dependent iterations; as part of k_finalize (128-thread CTAs, one per frame) the
//               256 frames of a batch needed two waves over the 148 SMs at 7 % warp occupancy (ncu r1x: 0.44 ms).  Warp
//               CTAs put all markers of the batch on the device at once: one chain latency instead of two.
//   k_board_batch: one warp per frame -- BoardDetector::detect on the frame's markers (when a board is armed).
#pragma once
#include "ab_device.cuh"

namespace ab {

__global__ void __launch_bounds__(128) k_finalize(Batch b) {
    __shared__ short s_src[MAX_CANDS];    // candidate index of the i-th decoded marker
    __shared__ short s_sorted[MAX_CANDS]; // decoded index at sorted position
    __shared__ float s_c[MAX_CANDS][8];
    __shared__ int s_id[MAX_CANDS];
    __shared__ uint8_t s_rm[MAX_CANDS];
    __shared__ short s_outpos[MAX_CANDS];
    __shared__ int s_n, s_nout;
    const int f = blockIdx.x, t = threadIdx.x;
    int nc = (int)b.n_cands[f];
    if (nc > b.cap_c) nc = b.cap_c;
    const CandRec* cands = b.cands + (size_t)f * b.cap_c;
    if (t == 0) {
        int n = 0;
        for (int i = 0; i < nc; i++)
            if (cands[i].id >= 0) s_src[n++] = (short)i;
        s_n = n;
    }
    __syncthreads();
    const int n = s_n;
    // stable rank by id (:417; SURVEY B.8)
    for (int i = t; i < n; i += blockDim.x) {
        int id = cands[s_src[i]].id;
        int rank = 0;
        for (int j = 0; j < n; j++) {
            int idj = cands[s_src[j]].id;
            rank += (idj < id) || (idj == id && j < i);
        }
        s_sorted[rank] = (short)i;
    }
    __syncthreads();
    for (int p = t; p < n; p += blockDim.x) {
        const CandRec& cr = cands[s_src[s_sorted[p]]];
        int nrot = cr.nrot & 3;
        // std::rotate(begin, begin + 4 - nRotations, end) (:364-366)
        for (int j = 0; j < 4; j++) {
            int sidx = (j + 4 - nrot) & 3;
            s_c[p][2 * j] = cr.refined[2 * sidx];
            s_c[p][2 * j + 1] = cr.refined[2 * sidx + 1];
        }
        s_id[p] = cr.id;
        s_rm[p] = 0;
    }
    __syncthreads();
    // duplicates (:421-430): adjacent equal ids -> remove the one with the smaller perimeter
    for (int p = t; p + 1 < n; p += blockDim.x) {
        if (s_id[p] == s_id[p + 1]) {
            if (perimeter4(s_c[p]) > perimeter4(s_c[p + 1])) s_rm[p + 1] = 1;
            else s_rm[p] = 1;
        }
    }
    __syncthreads();
    // border filter (:433-447): Point2f -> Point2i rounds (half to even)
    for (int p = t; p < n; p += blockDim.x) {
        for (int j = 0; j < 4; j++) {
            float x = s_c[p][2 * j], y = s_c[p][2 * j + 1];
            bool bad = !(isfinite(x) && isfinite(y));
            if (!bad) {
                int xi = __float2int_rn(x), yi = __float2int_rn(y);
                bad = !(xi >= b.vx0 && xi < b.vx1 && yi >= b.vy0 && yi < b.vy1);
            }
            if (bad) {
                s_rm[p] = 1;
                break;
            }
        }
    }
    __syncthreads();
    if (t == 0) {
        int o = 0;
        for (int p = 0; p < n; p++) s_outpos[p] = s_rm[p] ? (short)-1 : (short)o++;
        s_nout = o;
        b.n_markers[f] = (unsigned)o;
        atomicAdd(&b.cnt->n_markers_total, (unsigned long long)o);
    }
    __syncthreads();
    ab_marker* out = b.markers + (size_t)f * b.cap_c;
    for (int p = t; p < n; p += blockDim.x) {
        int o = s_outpos[p];
        if (o < 0) continue;
        ab_marker m;
        m.id = s_id[p];
        for (int j = 0; j < 8; j++) m.corners[j] = s_c[p][j];
        m.ssize = -1.f;
        m.pad_ = 0.f;
        m.has_pose = 0;
        for (int j = 0; j < 3; j++) m.rvec[j] = m.tvec[j] = 0.0;
        out[o] = m;
    }
}

// pose of every marker k_finalize kept (:450-467); launched only when a camera and a marker size were given (:450)
__global__ void __launch_bounds__(32) k_pose(Batch b) {
    const int f = blockIdx.y, slot = blockIdx.x * 32 + threadIdx.x;
    if (slot >= (int)b.n_markers[f]) return;
    ab_marker* m = b.markers + (size_t)f * b.cap_c + slot;
    float c[8];
#pragma unroll
    for (int j = 0; j < 8; j++) c[j] = m->corners[j];
    double r[3] = {0, 0, 0}, tv[3] = {0, 0, 0};
    int ok = 0;
    if (solve_pnp_marker(b.cam, c, b.marker_size, r, tv)) {
        if (b.set_y_perp) rotate_x_axis(r);
        ok = 1;
    }
    for (int j = 0; j < 3; j++) {
        m->rvec[j] = r[j];
        m->tvec[j] = tv[j];
    }
    m->has_pose = ok;
    m->ssize = b.marker_size;
}

// Marker::calculateExtrinsics for an array of markers (public worker)
__global__ void k_extrinsics(ab_marker* m, int n, Camera cam, float size, int set_y_perp) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double r[3] = {0, 0, 0}, tv[3] = {0, 0, 0};
    float c[8];
    for (int j = 0; j < 8; j++) c[j] = m[i].corners[j];
    bool ok = solve_pnp_marker(cam, c, size, r, tv);
    if (ok && set_y_perp) rotate_x_axis(r);
    for (int j = 0; j < 3; j++) {
        m[i].rvec[j] = r[j];
        m[i].tvec[j] = tv[j];
    }
    m[i].has_pose = ok;
    m[i].ssize = size;
}

// BoardDetector::detect (src/boarddetector.cpp:90-204) on every frame of a batch: ONE WARP per frame.  Lane 0 selects the
// frame's markers that belong to the configuration and stacks their corners (board_select_stack); the pose runs over the N
// stacked corners with the point loops lane-strided and butterfly sums (see PnpWarp), everything else computed identically by
// all lanes -- so every branch that reaches a shuffle depends only on values all lanes share (nb, a.pose, ok, the inlier count).
// Writes one ab_board per frame and the marker indices of the matched markers; ab_detect_board runs this kernel as a
// one-frame batch.
__global__ void __launch_bounds__(32) k_board_batch(Batch b, BoardArgs a) {
    const int f = blockIdx.x, lane = threadIdx.x;
    const int cap = b.cap_c;
    const int nm = min((int)b.n_markers[f], cap);
    float* obj = b.board_pts + (size_t)f * cap * BOARD_PTS_PER_MARKER;
    float* img = obj + 12 * (size_t)cap;
    float* obj2 = img + 8 * (size_t)cap;
    float* img2 = obj2 + 12 * (size_t)cap;
    int nb = 0;
    if (lane == 0)
        nb = board_select_stack(b.markers + (size_t)f * cap, nm, a.ids, a.corners, a.n_cfg, a.mpp, cap, obj, img,
                                b.board_slots + (size_t)f * cap);
    nb = __shfl_sync(0xFFFFFFFFu, nb, 0);
    __syncwarp();  // lane 0's stacked points are visible to the warp
    double r[3] = {0, 0, 0}, t[3] = {0, 0, 0};
    bool ok = false;
    if (nb > 0 && a.pose) {
        const int N = 4 * nb;
        ok = solve_pnp_planar_t<PnpWarp>(a.cam, obj, img, N, r, t);
        if (ok && a.repj_err_thres > 0) {  // reprojection-outlier re-solve (:172-194)
            double R[9];
            rodrigues_to_mat(r, R);
            int m = 0;
            for (int n = 0; n < N; n++) {  // order-preserving compaction of the inliers: every lane counts, lane 0 writes
                double X = obj[3 * n], Y = obj[3 * n + 1], Z = obj[3 * n + 2];
                double x = R[0] * X + R[1] * Y + R[2] * Z + t[0], y = R[3] * X + R[4] * Y + R[5] * Z + t[1], z = R[6] * X + R[7] * Y + R[8] * Z + t[2];
                z = z ? 1. / z : 1.;
                double u, v;
                distort_norm_to_px(a.cam, x * z, y * z, &u, &v);
                float du = (float)u - img[2 * n], dv = (float)v - img[2 * n + 1];  // projectPoints writes Point2f
                float err = (float)sqrt((double)du * du + (double)dv * dv);
                if (err < a.repj_err_thres) {
                    if (lane == 0) {
                        AB_BOUND(m < 4 * cap);
                        for (int c = 0; c < 3; c++) obj2[3 * m + c] = obj[3 * n + c];
                        img2[2 * m] = img[2 * n];
                        img2[2 * m + 1] = img[2 * n + 1];
                    }
                    m++;
                }
            }
            __syncwarp();
            ok = solve_pnp_planar_t<PnpWarp>(a.cam, obj2, img2, m, r, t);
        }
        if (ok && a.set_y_perp) rotate_x_axis(r);
    }
    if (lane == 0) {
        ab_board o;
        o.n_markers = nb;
        o.has_pose = ok ? 1 : 0;
        o.prob = nb > 0 && a.pose ? (float)nb / (float)a.n_cfg : 0.f;  // "return 0" without camera / information (:117-130)
        o.ssize = a.ssize;
        for (int i = 0; i < 3; i++) {
            o.rvec[i] = r[i];
            o.tvec[i] = t[i];
        }
        b.boards[f] = o;
    }
}

}  // namespace ab
