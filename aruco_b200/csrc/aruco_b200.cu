// libaruco_b200.so -- context management and the C ABI declared in include/aruco_b200.h.
// Everything computational happens in the kernels of k_*.cuh on the device; this file only sizes buffers,
// moves frames/results and launches.  There is deliberately no host implementation of any stage.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <algorithm>
#include <string>
#include <vector>

#include "ab_device.cuh"
#include "k_threshold.cuh"
#include "k_threshold_pair.cuh"
#include "k_threshold_tma.cuh"
#include "k_canny.cuh"
#include "k_contours.cuh"
#include "k_polygon.cuh"
#include "k_decode.cuh"
#include "k_render.cuh"
#include "k_refine.cuh"
#include "k_finalize.cuh"
#include "k_calib.cuh"

using namespace ab;

constexpr int WALKER_CTAS_PER_SM = 8;  // persistent grids of k_trace<false> and k_trace<true>
// d_counters / h_counters: one Counters, then the per-frame n_quads, n_cands and n_markers arrays (maxB entries each)
constexpr size_t FRAME_COUNTS_OFFSET = sizeof(Counters);

#ifndef AB_SOURCE_HASH
#define AB_SOURCE_HASH "unknown"
#endif
// "src:" = first 16 hex digits of sha256 over the product sources (Makefile SRCHASH; tests/conftest.py checks it)
#define AB_VERSION "aruco_b200 0.2 (sm_100a) src:" AB_SOURCE_HASH

struct ab_context {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;       // every kernel / copy of this context runs here (private, non-blocking)
    bool own_stream = true;
    cudaStream_t user_stream = nullptr;  // ab_set_stream: the caller's stream; each enqueue is ordered after it
    bool has_user_stream = false;
    cudaStream_t copy_stream = nullptr;
    uint2* d_trace_rec = nullptr;       // strips of k_trace<true>'s lanes (k_contours.cuh), grown on demand
    size_t trace_rec_bytes = 0;
    unsigned rec_ctas = 0, rec_half = 0;
    size_t trace_rec_budget = (size_t)6 << 30;  // more lanes than this pays for are not launched
    ab_params params;
    std::string err;
    // reserved geometry
    int W = 0, H = 0, maxB = 0, capQ = 0, capC = 0, S_alloc = 0;
    long long capStartsPF = 0, capPoolPF = 0;
    unsigned capContoursPF = 16384;
    // device buffers
    uint8_t* d_grey[2] = {nullptr, nullptr};
    size_t grey_bytes = 0;
    uint8_t* d_bgr = nullptr;
    size_t bgr_bytes = 0;
    uint8_t* d_thres = nullptr;
    uint32_t *d_bits = nullptr, *d_bits2 = nullptr;
    uint2* d_starts = nullptr;
    ContourRec* d_contours = nullptr;
    uint32_t* d_pool = nullptr;
    LongRec* d_longq = nullptr;
    uint8_t* d_walk_lut = nullptr;
    unsigned capLongPF = 8192;
    QuadRec* d_quads = nullptr;
    CandRec* d_cands = nullptr;
    uint8_t* d_canon = nullptr;
    CandAux* d_aux = nullptr;
    unsigned short* d_hist = nullptr;
    ab_marker* d_markers = nullptr;
    uint8_t* d_counters = nullptr;  // Counters + 3*maxB uints
    size_t counters_bytes = 0;
    // HRM dictionary
    uint64_t* d_dict_bits = nullptr;
    uint32_t* d_dict_ordids = nullptr;
    int32_t* d_dict_ordpos = nullptr;
    int32_t* d_dict_tree = nullptr;
    HrmDict dict{};
    bool have_dict = false;
    // host callback decoder
    ab_decoder_fn cb = nullptr;
    void* cb_user = nullptr;
    // pinned host staging
    ab_marker* h_markers = nullptr;
    size_t h_markers_bytes = 0;
    uint8_t* h_counters = nullptr;
    // last batch
    Batch last{};
    bool have_last = false;
    int last_n = 0;
    // timing
    bool timing = false;
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t kev[13] = {};  // boundaries: threshold|scan|trace|trace_long|emit|polygon|filter|sample|identify|refine|finalize|board
    cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};
    // Two batches in flight: a second, library-owned context (`twin`) carries the second set of per-batch buffers and
    // a private stream, so ab_enqueue_batch_device may be called again before ab_fetch_results and the kernels of
    // batch n+1 run under the latency-bound tail of batch n.  Results come back in enqueue order.
    ab_context* twin = nullptr;
    ab_context* owner = nullptr;   // set in the twin: errors are reported through the owner
    int pending[2] = {0, 0};       // FIFO of un-fetched batches: 0 = this context, 1 = the twin
    int n_pending = 0;
    int cur = 0;                   // which of the two the state getters read (last enqueued or fetched)
    bool worker_call = false;      // inside ab_threshold (thresHold never erodes: the u8 image must be written)
    void* d_scratch = nullptr;     // grow-only device scratch of the small per-call workers (board pose)
    size_t scratch_bytes = 0;
    double* h_scratch = nullptr;   // pinned result slot of those workers
    cudaEvent_t ev_in = nullptr;   // orders the twin's stream after the caller's stream at enqueue time
    // capacities the caller chose in ab_reserve (0 = defaults); kept across automatic re-reservations
    int userQ = 0, userC = 0;
    long long userStarts = 0, userPoints = 0;
    // armed board configuration (ab_set_board): the device arrays belong to the owner; get_twin copies `board` to the twin
    int32_t* d_board_ids = nullptr;
    float* d_board_corners = nullptr;
    BoardArgs board{};
    bool have_board = false;
    // per-batch board outputs of k_board_batch, sized maxB x capC by the first batch that runs with a board armed
    ab_board* d_boards = nullptr;
    int32_t* d_board_slots = nullptr;
    float* d_board_pts = nullptr;
    int board_frames = 0, board_capc = 0;
    ab_board* h_boards = nullptr;  // pinned staging of fetch_into
    size_t h_boards_bytes = 0;
    int32_t* h_board_slots = nullptr;
    size_t h_board_slots_bytes = 0;
    // owner side: the boards of the batch last returned by ab_fetch_results / ab_detect_batch(_bgr), all chunks of it
    bool res_board = false;          // every chunk of that batch ran with a board armed
    bool res_board_markers = false;  // and its markers were fetched, so that the matched markers are known
    std::vector<ab_board> res_boards;
    std::vector<int32_t> res_off;    // [frames + 1]: frame f's matched markers are res_markers[res_off[f] .. res_off[f + 1])
    std::vector<ab_marker> res_markers;
};

// RAII device temporary of the secondary entry points: freed on every return path
struct DevBuf {
    void* p = nullptr;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() {
        if (p) cudaFree(p);
    }
    cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, bytes ? bytes : 1); }
    template <class T>
    T* as() const {
        return (T*)p;
    }
};

static int set_err(ab_context* c, int code, const char* fmt, ...) {
    if (c && c->owner) c = c->owner;
    if (c) {
        char buf[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof(buf), fmt, ap);
        va_end(ap);
        c->err = buf;
    }
    return code;
}

#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess)                                                                           \
            return set_err(ctx, AB_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

static int ensure_scratch(ab_context* ctx, size_t bytes) {
    if (!ctx->h_scratch) CK(cudaMallocHost(&ctx->h_scratch, 64 * sizeof(double)));
    if (ctx->scratch_bytes >= bytes) return AB_OK;
    if (ctx->d_scratch) cudaFree(ctx->d_scratch);
    ctx->d_scratch = nullptr;
    ctx->scratch_bytes = 0;
    bytes = (bytes + 4095) & ~(size_t)4095;
    CK(cudaMalloc(&ctx->d_scratch, bytes));
    ctx->scratch_bytes = bytes;
    return AB_OK;
}

static void free_buffers(ab_context* c) {
    auto F = [](auto*& p) {
        if (p) cudaFree(p);
        p = nullptr;
    };
    F(c->d_grey[0]);
    F(c->d_grey[1]);
    F(c->d_bgr);
    F(c->d_thres);
    F(c->d_bits);
    F(c->d_bits2);
    F(c->d_starts);
    F(c->d_contours);
    F(c->d_pool);
    F(c->d_longq);
    F(c->d_trace_rec);
    c->trace_rec_bytes = 0;
    F(c->d_quads);
    F(c->d_cands);
    F(c->d_canon);
    F(c->d_aux);
    F(c->d_hist);
    F(c->d_markers);
    F(c->d_counters);
    F(c->d_boards);
    F(c->d_board_slots);
    F(c->d_board_pts);
    c->board_frames = c->board_capc = 0;
    if (c->h_boards) cudaFreeHost(c->h_boards);
    c->h_boards = nullptr;
    c->h_boards_bytes = 0;
    if (c->h_board_slots) cudaFreeHost(c->h_board_slots);
    c->h_board_slots = nullptr;
    c->h_board_slots_bytes = 0;
    if (c->h_markers) cudaFreeHost(c->h_markers);
    c->h_markers = nullptr;
    c->h_markers_bytes = 0;
    if (c->h_counters) cudaFreeHost(c->h_counters);
    c->h_counters = nullptr;
    c->grey_bytes = c->bgr_bytes = 0;
    c->W = c->H = c->maxB = 0;
    c->have_last = false;
}

extern "C" {

const char* ab_version(void) { return AB_VERSION; }

const char* ab_last_error(const ab_context* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int ab_default_params(ab_params* p) {
    if (!p) return AB_E_INVALID;
    memset(p, 0, sizeof(*p));
    p->thres_method = AB_THRES_ADAPTIVE;
    p->thres_param1 = 7;
    p->thres_param2 = 7;
    p->corner_method = AB_CORNER_LINES;
    p->min_size = 0.04f;
    p->max_size = 0.5f;
    p->warp_size = 56;
    p->border_dist = 0.025f;
    p->locked_corners = 0;
    p->erosion = 0;
    p->decoder = AB_DECODER_FIDUCIDAL;
    p->set_y_perpendicular = 0;
    p->thres_param1_range = 0;
    return AB_OK;
}

int ab_create(int device, ab_context** out) {
    if (!out) return AB_E_INVALID;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || device < 0 || device >= ndev) return AB_E_NO_DEVICE;
    ab_context* ctx = new ab_context();
    ctx->device = device;
    ab_default_params(&ctx->params);
    if (cudaSetDevice(device) != cudaSuccess) {
        delete ctx;
        return AB_E_NO_DEVICE;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete ctx;
        return AB_E_CUDA;
    }
    {  // step tables of the border walkers (ab_trace.cuh)
        std::vector<uint8_t> lut(2 * WALK_LUT_SIZE);
        for (uint32_t i = 0; i < (uint32_t)WALK_LUT_SIZE; i++) {
            lut[i] = walk_lut_fw_entry(i);
            lut[WALK_LUT_SIZE + i] = walk_lut_bw_entry(i);
        }
        if (cudaMalloc(&ctx->d_walk_lut, lut.size()) != cudaSuccess ||
            cudaMemcpyAsync(ctx->d_walk_lut, lut.data(), lut.size(), cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess ||
            cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
            cudaGetLastError();
            if (ctx->d_walk_lut) cudaFree(ctx->d_walk_lut);
            cudaStreamDestroy(ctx->stream);
            cudaStreamDestroy(ctx->copy_stream);
            delete ctx;
            return AB_E_CUDA;
        }
    }
    // capacity of the parked-walk queue per frame (tests shrink it to exercise the finish-in-place path)
    if (const char* e = getenv("ARUCO_B200_CAP_LONG")) ctx->capLongPF = (unsigned)std::max(1, atoi(e));
    if (const char* e = getenv("ARUCO_B200_TRACE_REC_MB")) ctx->trace_rec_budget = (size_t)std::max(1, atoi(e)) << 20;
    for (int i = 0; i < 6; i++) cudaEventCreate(&ctx->ev[i]);
    for (int i = 0; i < 13; i++) cudaEventCreate(&ctx->kev[i]);
    for (int i = 0; i < 2; i++) {
        cudaEventCreateWithFlags(&ctx->ev_h2d[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&ctx->ev_done[i], cudaEventDisableTiming);
    }
    cudaEventCreateWithFlags(&ctx->ev_in, cudaEventDisableTiming);
    *out = ctx;
    return AB_OK;
}

void ab_destroy(ab_context* ctx) {
    if (!ctx) return;
    if (ctx->twin) {
        ab_destroy(ctx->twin);
        ctx->twin = nullptr;
    }
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    free_buffers(ctx);
    if (ctx->d_walk_lut) cudaFree(ctx->d_walk_lut);
    auto F = [](auto*& p) {
        if (p) cudaFree(p);
        p = nullptr;
    };
    if (!ctx->owner) {  // the twin borrows the owner's dictionary
        F(ctx->d_dict_bits);
        F(ctx->d_dict_ordids);
        F(ctx->d_dict_ordpos);
        F(ctx->d_dict_tree);
        F(ctx->d_board_ids);
        F(ctx->d_board_corners);
    }
    if (ctx->ev_in) cudaEventDestroy(ctx->ev_in);
    if (ctx->d_scratch) cudaFree(ctx->d_scratch);
    if (ctx->h_scratch) cudaFreeHost(ctx->h_scratch);
    for (int i = 0; i < 6; i++)
        if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    for (int i = 0; i < 13; i++)
        if (ctx->kev[i]) cudaEventDestroy(ctx->kev[i]);
    for (int i = 0; i < 2; i++) {
        if (ctx->ev_h2d[i]) cudaEventDestroy(ctx->ev_h2d[i]);
        if (ctx->ev_done[i]) cudaEventDestroy(ctx->ev_done[i]);
    }
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    delete ctx;
}

int ab_set_params(ab_context* ctx, const ab_params* p) {
    if (!ctx || !p) return AB_E_INVALID;
    // the reference's CV_Asserts: setMinMaxSize (cpp:1031-1038), setWarpSize (cpp:1047-1051)
    if (!(p->min_size > 0 && p->min_size <= 1) || !(p->max_size > 0 && p->max_size <= 1) || !(p->min_size < p->max_size))
        return set_err(ctx, AB_E_INVALID, "setMinMaxSize: need 0 < min < max <= 1");
    if (p->warp_size < 10 || p->warp_size > MAX_WARP_SIZE)
        return set_err(ctx, AB_E_INVALID, "setWarpSize: need 10 <= size <= %d", MAX_WARP_SIZE);
    if (p->thres_method < 0 || p->thres_method > 2) return set_err(ctx, AB_E_INVALID, "bad threshold method");
    if (p->corner_method < 0 || p->corner_method > 3) return set_err(ctx, AB_E_INVALID, "bad corner refinement method");
    if (p->decoder < 0 || p->decoder > 2) return set_err(ctx, AB_E_INVALID, "bad decoder kind");
    if (p->thres_param1_range < 0 || p->thres_param1_range > 7) return set_err(ctx, AB_E_INVALID, "threshold param range outside 0..7");
    ctx->params = *p;
    return AB_OK;
}

int ab_get_params(const ab_context* ctx, ab_params* p) {
    if (!ctx || !p) return AB_E_INVALID;
    *p = ctx->params;
    return AB_OK;
}

int ab_set_stream(ab_context* ctx, void* s) {
    if (!ctx) return AB_E_INVALID;
    // The handle is used as given: NULL is the caller's legacy default stream (handle 0), which is what torch reports for
    // its default stream.  The library keeps launching on its own streams (one per in-flight batch, so that two batches can
    // overlap); every enqueue first records an event on the caller's stream and makes its stream wait for it.
    ctx->user_stream = (cudaStream_t)s;
    ctx->has_user_stream = true;
    return AB_OK;
}

int ab_set_decoder_callback(ab_context* ctx, ab_decoder_fn fn, void* user) {
    if (!ctx) return AB_E_INVALID;
    ctx->cb = fn;
    ctx->cb_user = user;
    return AB_OK;
}

int ab_enable_timing(ab_context* ctx, int enable) {
    if (!ctx) return AB_E_INVALID;
    ctx->timing = enable != 0;
    return AB_OK;
}

int ab_load_hrm_dictionary(ab_context* ctx, int n, int count, const uint8_t* bits, int tau0, float rate) {
    if (!ctx || !bits || n < 1 || n > 8 || count < 1 || count > 16383) return set_err(ctx, AB_E_INVALID, "bad dictionary");
    cudaSetDevice(ctx->device);
    std::vector<uint64_t> b0(count);
    std::vector<uint32_t> id0(count);
    for (int i = 0; i < count; i++) {
        uint64_t rb[4];
        uint32_t ids[4];
        hrm_rotations(bits + (size_t)i * n * n, n, rb, ids);
        b0[i] = rb[0];
        id0[i] = ids[0];
    }
    // BalancedBinaryTree::loadDictionary (highlyreliablemarkers.cpp:387-476): the search structure is data,
    // built once on the host; the lookups run on the device (k_decode.cuh hrm_decode).
    std::vector<std::pair<uint32_t, uint32_t>> order(count);
    for (int i = 0; i < count; i++) order[i] = {id0[i], (uint32_t)i};
    std::sort(order.begin(), order.end());
    unsigned sz = (unsigned)count, levels = 0;
    while (powf(2.f, (float)levels) <= (float)sz) levels++;
    std::vector<char> visited(sz, 0);
    unsigned root = sz / 2;
    visited[root] = 1;
    std::vector<std::pair<unsigned, unsigned>> intervals;
    intervals.push_back({0u, root});
    intervals.push_back({root, sz});
    std::vector<int32_t> tree(2 * (size_t)sz, 0);
    tree[2 * root] = !visited[(0 + root) / 2] ? (int)((0 + root) / 2) : -1;
    tree[2 * root + 1] = !visited[(root + sz) / 2] ? (int)((root + sz) / 2) : -1;
    for (unsigned lv = 1; lv < levels; lv++) {
        size_t nint = intervals.size();
        for (size_t j = 0; j < nint; j++) {
            unsigned lo = intervals.back().first, hi = intervals.back().second;
            intervals.pop_back();
            unsigned center = (hi + lo) / 2;
            if (!visited[center]) visited[center] = 1;
            else continue;
            unsigned lc = (lo + center) / 2, hc = (center + hi) / 2;
            if (!visited[lc]) {
                intervals.insert(intervals.begin(), {lo, center});
                tree[2 * center] = (int)lc;
            } else tree[2 * center] = -1;
            if (!visited[hc]) {
                intervals.insert(intervals.begin(), {center, hi});
                tree[2 * center + 1] = (int)hc;
            } else tree[2 * center + 1] = -1;
        }
    }
    std::vector<uint32_t> ordids(count);
    std::vector<int32_t> ordpos(count);
    for (int i = 0; i < count; i++) {
        ordids[i] = order[i].first;
        ordpos[i] = (int32_t)order[i].second;
    }
    auto F = [](auto*& p) {
        if (p) cudaFree(p);
        p = nullptr;
    };
    if (ctx->twin) cudaStreamSynchronize(ctx->twin->stream);  // it may still be decoding with the old dictionary
    ctx->have_dict = false;
    F(ctx->d_dict_bits);
    F(ctx->d_dict_ordids);
    F(ctx->d_dict_ordpos);
    F(ctx->d_dict_tree);
    CK(cudaMalloc(&ctx->d_dict_bits, sizeof(uint64_t) * count));
    CK(cudaMalloc(&ctx->d_dict_ordids, sizeof(uint32_t) * count));
    CK(cudaMalloc(&ctx->d_dict_ordpos, sizeof(int32_t) * count));
    CK(cudaMalloc(&ctx->d_dict_tree, sizeof(int32_t) * 2 * count));
    CK(cudaMemcpyAsync(ctx->d_dict_bits, b0.data(), sizeof(uint64_t) * count, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_dict_ordids, ordids.data(), sizeof(uint32_t) * count, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_dict_ordpos, ordpos.data(), sizeof(int32_t) * count, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_dict_tree, tree.data(), sizeof(int32_t) * 2 * count, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));  // the host vectors go out of scope
    ctx->dict.bits = ctx->d_dict_bits;
    ctx->dict.ids = nullptr;
    ctx->dict.ord_ids = ctx->d_dict_ordids;
    ctx->dict.ord_pos = ctx->d_dict_ordpos;
    ctx->dict.tree = ctx->d_dict_tree;
    ctx->dict.root = (int)root;
    ctx->dict.count = count;
    ctx->dict.n = n;
    ctx->dict.correction = (int)(rate * (float)((tau0 - 1) / 2));  // highlyreliablemarkers.cpp:318
    ctx->have_dict = true;
    return AB_OK;
}

static int reserve_impl(ab_context* ctx, int width, int height, int max_batch) {
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    free_buffers(ctx);  // zeroes W/H/maxB: a failed reservation leaves a context that re-reserves on the next call
    const int capQ = ctx->userQ > 0 ? std::min(ctx->userQ, MAX_QUADS) : MAX_QUADS;
    const int capC = ctx->userC > 0 ? std::min(ctx->userC, MAX_CANDS) : 512;
    const long long px = (long long)width * height;
    const long long capS = ctx->userStarts > 0 ? ctx->userStarts : std::max(px / 8, 65536LL);
    long long capP = ctx->userPoints > 0 ? ctx->userPoints : std::max(px / 4, 65536LL);
    if (capP * max_batch > 0xFFFFFFF0LL) capP = 0xFFFFFFF0LL / max_batch;
    const int S_alloc = std::max(ctx->params.warp_size, 56);
    const size_t B = (size_t)max_batch;
    const size_t bw = bit_image_words(width, height);
    const size_t counters_bytes = FRAME_COUNTS_OFFSET + 3 * B * sizeof(unsigned);
    cudaError_t e = cudaSuccess;
    auto A = [&](auto** p, size_t bytes) {
        if (e == cudaSuccess) e = cudaMalloc(p, bytes);
    };
    A(&ctx->d_thres, B * px);
    A(&ctx->d_bits, B * bw * 4);
    A(&ctx->d_bits2, B * bw * 4);
    A(&ctx->d_starts, B * capS * sizeof(uint2));
    A(&ctx->d_contours, B * ctx->capContoursPF * sizeof(ContourRec));
    A(&ctx->d_pool, B * capP * 4);
    A(&ctx->d_longq, B * ctx->capLongPF * sizeof(LongRec));
    A(&ctx->d_quads, B * capQ * sizeof(QuadRec));
    A(&ctx->d_cands, B * capC * sizeof(CandRec));
    A(&ctx->d_canon, B * capC * (size_t)S_alloc * S_alloc);
    A(&ctx->d_aux, B * capC * sizeof(CandAux));
    A(&ctx->d_hist, B * capC * 256 * sizeof(unsigned short));
    A(&ctx->d_markers, B * capC * sizeof(ab_marker));
    A(&ctx->d_counters, counters_bytes);
    if (e == cudaSuccess) e = cudaMallocHost(&ctx->h_counters, counters_bytes);
    // the zero frame around the packed image is written once; the kernels only write inside it
    if (e == cudaSuccess) e = cudaMemsetAsync(ctx->d_bits, 0, B * bw * 4, ctx->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(ctx->d_bits2, 0, B * bw * 4, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        cudaGetLastError();
        free_buffers(ctx);
        return set_err(ctx, AB_E_CUDA, "ab_reserve(%dx%d x%d): %s", width, height, max_batch, cudaGetErrorString(e));
    }
    ctx->W = width;
    ctx->H = height;
    ctx->maxB = max_batch;
    ctx->capQ = capQ;
    ctx->capC = capC;
    ctx->capStartsPF = capS;
    ctx->capPoolPF = capP;
    ctx->S_alloc = S_alloc;
    ctx->counters_bytes = counters_bytes;
    return AB_OK;
}

int ab_reserve(ab_context* ctx, int width, int height, int max_batch, int max_quads, int max_cands,
               int64_t max_starts_pf, int64_t max_points_pf) {
    if (!ctx || width < 8 || height < 8 || width > 16384 || height > 16384 || max_batch < 1)
        return set_err(ctx, AB_E_INVALID, "ab_reserve: bad geometry %dx%d x%d", width, height, max_batch);
    if (ctx->n_pending) return set_err(ctx, AB_E_STATE, "ab_reserve: %d batch(es) in flight, fetch them first", ctx->n_pending);
    // the caller's capacities are remembered: automatic re-reservations (larger batch, other warp size) keep them
    ctx->userQ = max_quads;
    ctx->userC = max_cands;
    ctx->userStarts = max_starts_pf;
    ctx->userPoints = max_points_pf;
    if (ctx->twin) free_buffers(ctx->twin);  // re-reserved with the new capacities when it is next used
    return reserve_impl(ctx, width, height, max_batch);
}

// threshold images per frame (setThresholdParamRange, cpp:322-334); CANNY ignores the parameters: one image
static int n_thres_images(const ab_params& P) { return P.thres_method == AB_THRES_CANNY ? 1 : 2 * P.thres_param1_range + 1; }

static int ensure_reserved(ab_context* ctx, int W, int H, int nB) {
    if (ctx->W == W && ctx->H == H && ctx->maxB >= nB && ctx->S_alloc >= ctx->params.warp_size) return AB_OK;
    int B = (ctx->W == W && ctx->H == H) ? std::max(ctx->maxB, nB) : nB;
    return reserve_impl(ctx, W, H, B);
}

static Camera make_camera(const float* K, const float* D) {
    Camera c;
    memset(&c, 0, sizeof(c));
    if (K) {
        c.has_K = 1;
        c.fxf = K[0];
        c.cxf = K[2];
        c.fyf = K[4];
        c.cyf = K[5];
        c.fx = K[0];
        c.cx = K[2];
        c.fy = K[4];
        c.cy = K[5];
    }
    if (D) {
        c.has_D = 1;
        c.k1 = D[0];
        c.k2 = D[1];
        c.p1 = D[2];
        c.p2 = D[3];
        c.k3 = D[4];
        c.zero_D = D[0] == 0.f && D[1] == 0.f && D[2] == 0.f && D[3] == 0.f && D[4] == 0.f;
    }
    return c;
}

static int launch_threshold(ab_context* ctx, const Batch& b, int method, double p1, double p2, int out_mul = 1, int out_off = 0,
                            cudaStream_t st_in = nullptr) {
    cudaStream_t st = st_in ? st_in : ctx->stream;
    if (method == AB_THRES_ADAPTIVE) {
        // thresHold: ensure an odd block size >= 3 (src/markerdetector.cpp:657-660)
        if (p1 < 3) p1 = 3;
        else if (((int)p1) % 2 != 1) p1 = (int)(p1 + 1);
        int k = (int)p1;
        if (k > 63) return set_err(ctx, AB_E_INVALID, "adaptive threshold block size %d > 63 not supported", k);
        double fl = floor(p2);
        int idelta = (int)std::max(-300.0, std::min(300.0, fl));
        ThrArgs a;
        a.grey = b.grey;
        a.grey_row = b.grey_row;
        a.grey_frame = b.grey_frame;
        a.thres = b.thres;
        a.bits = b.bits;
        a.bits_words = b.bits_words;
        a.W = b.W;
        a.H = b.H;
        a.wpr = b.wpr;
        a.k = k;
        a.idelta = idelta;
        a.TWo = 480;
        a.RH = k <= 9 ? 64 : 128;
        int r = k / 2;
        a.R4 = (r + 3) & ~3;
        a.aligned4 = ((((uintptr_t)b.grey) | b.grey_row | b.grey_frame) & 3) == 0;
        a.out_mul = out_mul;
        a.out_off = out_off;
        a.skip_u8 = ctx->params.erosion != 0 && !ctx->worker_call;  // k_erode writes the (eroded) u8 image
        int nth = (a.TWo + 2 * a.R4) / 4;
        nth = (nth + 31) & ~31;
        size_t SPAN = 4 * (size_t)nth;
        size_t smem = (((size_t)k * SPAN + 15) & ~(size_t)15) + 4 * SPAN + nth;
        dim3 grid((b.W + a.TWo - 1) / a.TWo, (b.H + a.RH - 1) / a.RH, b.B);
        if (!launch_threshold_tma(a, b.B, st) && !launch_threshold_pair(a, b.B, st) && !launch_threshold_fast(a, b.B, st))
            k_threshold_adaptive<<<grid, nth, smem, st>>>(a);
    } else if (method == AB_THRES_FIXED) {
        int thr = (int)floor(p1);
        k_threshold_fixed<<<ctx->sm_count * 8, 256, 0, st>>>(b.grey, b.grey_row, b.grey_frame, b.thres, b.bits, b.bits_words,
                                                              b.W, b.H, b.wpr, thr, 0, b.B, out_mul, out_off);
    } else {
        // CANNY (src/markerdetector.cpp:669): cv::Canny(grey, out, 10, 220).  The map (0/1/2) is built in the
        // virtual frames' thres slots; hysteresis passes repeat until a group of passes changes no tile -- the
        // only place on the path where the host looks at a device flag mid-batch (the edge set is data dependent).
        uint8_t* map = b.thres;
        dim3 g1((b.W + 31) / 32, (b.H + 7) / 8, b.B);
        k_canny_nms<<<g1, dim3(32, 8), 0, st>>>(b.grey, b.grey_row, b.grey_frame, map, b.W, b.H, 10, 220);
        unsigned int* d_changed = &b.cnt->canny_changed;
        dim3 g2((b.W + 31) / 32, (b.H + 31) / 32, b.B);
        for (int group = 0; group < 4096; group++) {
            CK(cudaMemsetAsync(d_changed, 0, sizeof(unsigned), st));
            for (int pass = 0; pass < 4; pass++) k_canny_hyst<<<g2, 256, 0, st>>>(map, b.W, b.H, d_changed);
            unsigned h_changed = 0;
            CK(cudaMemcpyAsync(&h_changed, d_changed, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            if (!h_changed) break;
        }
        k_canny_finish<<<ctx->sm_count * 8, 256, 0, st>>>(b.thres, b.bits, b.bits_words, b.W, b.H, b.wpr, b.B, out_mul, out_off);
    }
    CK(cudaGetLastError());
    return AB_OK;
}

__global__ void k_set_ids(Batch b, const int2* idrot) {
    int f = blockIdx.y, ci = blockIdx.x * blockDim.x + threadIdx.x;
    if (ci >= (int)b.n_cands[f]) return;
    int2 v = idrot[(size_t)f * b.cap_c + ci];
    b.cands[(size_t)f * b.cap_c + ci].id = v.x;
    b.cands[(size_t)f * b.cap_c + ci].nrot = v.y;
}

// cvtColor(BGR2GRAY) of OpenCV 4.x: (3735 B + 19235 G + 9798 R + 16384) >> 15   (SURVEY A.11).  A thread converts 4
// consecutive pixels of a row (W % 4 == 0: three 32-bit loads, one 32-bit store; else bytes); the row/frame split is done
// once per thread group of a row, not per pixel.
__global__ void k_bgr2grey(const uint8_t* bgr, size_t row, size_t frame, uint8_t* grey, int W, int H, int B) {
    const int qpr = (W + 3) / 4;  // 4-pixel groups per row
    const size_t total = (size_t)qpr * H * B;
    const bool vec = (W & 3) == 0 && (row & 3) == 0 && (frame & 3) == 0 && (((uintptr_t)bgr | (uintptr_t)grey) & 3) == 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const unsigned line = (unsigned)(i / (unsigned)qpr);  // < H * B < 2^32
        const int q = (int)(i - (size_t)line * qpr);
        const int f = (int)(line / (unsigned)H), y = (int)(line - (unsigned)f * H);
        const uint8_t* p = bgr + (size_t)f * frame + (size_t)y * row + 12 * (size_t)q;
        uint8_t* g = grey + ((size_t)f * H + y) * W + 4 * (size_t)q;
        if (vec) {
            const uint32_t w0 = *reinterpret_cast<const uint32_t*>(p), w1 = *reinterpret_cast<const uint32_t*>(p + 4),
                           w2 = *reinterpret_cast<const uint32_t*>(p + 8);
            auto lum = [](uint32_t bb, uint32_t gg, uint32_t rr) { return (3735u * bb + 19235u * gg + 9798u * rr + 16384u) >> 15; };
            const uint32_t g0 = lum(w0 & 255, (w0 >> 8) & 255, (w0 >> 16) & 255), g1 = lum(w0 >> 24, w1 & 255, (w1 >> 8) & 255);
            const uint32_t g2 = lum((w1 >> 16) & 255, w1 >> 24, w2 & 255), g3 = lum((w2 >> 8) & 255, (w2 >> 16) & 255, w2 >> 24);
            *reinterpret_cast<uint32_t*>(g) = g0 | (g1 << 8) | (g2 << 16) | (g3 << 24);
        } else {
            for (int k = 0; k < 4 && 4 * q + k < W; k++)
                g[k] = (uint8_t)((3735 * p[3 * k] + 19235 * p[3 * k + 1] + 9798 * p[3 * k + 2] + 16384) >> 15);
        }
    }
}

// n frames of n_t threshold images each: the per-frame capacities of the append lists count the n * n_t virtual frames
static int fill_batch(ab_context* ctx, Batch& b, const uint8_t* dgrey, size_t row, size_t frame, int n, int n_t, const float* K,
                      const float* D, float marker_size) {
    const ab_params& P = ctx->params;
    const int nv = n * n_t;
    memset(&b, 0, sizeof(b));
    b.W = ctx->W;
    b.H = ctx->H;
    b.B = n;
    b.n_t = n_t;
    b.wpr = bit_words_per_row(ctx->W);
    b.bits_words = bit_image_words(ctx->W, ctx->H);
    b.grey = dgrey;
    b.grey_row = row;
    b.grey_frame = frame;
    b.thres = ctx->d_thres;
    b.bits = ctx->d_bits;
    b.bits2 = ctx->d_bits2;
    b.starts = ctx->d_starts;
    b.cap_starts = (unsigned long long)ctx->capStartsPF * nv;
    b.contours = ctx->d_contours;
    b.cap_contours = ctx->capContoursPF * (unsigned)nv;
    b.longq = ctx->d_longq;
    b.cap_long = ctx->capLongPF * (unsigned)nv;
    b.walk_lut = ctx->d_walk_lut;
    b.pool = ctx->d_pool;
    b.cap_pool = (unsigned long long)ctx->capPoolPF * nv;
    b.quads = ctx->d_quads;
    b.cap_q = ctx->capQ;
    b.cands = ctx->d_cands;
    b.cap_c = ctx->capC;
    b.canon = ctx->d_canon;
    b.aux = ctx->d_aux;
    b.hist = ctx->d_hist;
    b.markers = ctx->d_markers;
    b.cnt = (Counters*)ctx->d_counters;
    b.n_quads = (unsigned*)(ctx->d_counters + FRAME_COUNTS_OFFSET);
    b.n_cands = b.n_quads + ctx->maxB;
    b.n_markers = b.n_cands + ctx->maxB;
    // contour length limits (src/markerdetector.cpp:500-501): f32 product truncated to int
    int mx = std::max(ctx->W, ctx->H);
    b.min_len = (int)(P.min_size * (float)mx * 4.f);
    b.max_len = (int)(P.max_size * (float)mx * 4.f);
    b.S = P.warp_size;
    b.decoder = P.decoder;
    b.corner_method = P.corner_method;
    b.subpix_win = (int)P.thres_param1;
    b.locked = P.locked_corners;
    b.set_y_perp = P.set_y_perpendicular;
    // valid region (src/markerdetector.cpp:433-434): Point*float rounds half-to-even
    float bd = P.border_dist, ob = 1.0f - bd;
    int x0 = (int)lrintf((float)ctx->W * bd), y0 = (int)lrintf((float)ctx->H * bd);
    int x1 = (int)lrintf((float)ctx->W * ob), y1 = (int)lrintf((float)ctx->H * ob);
    b.vx0 = std::min(x0, x1);
    b.vy0 = std::min(y0, y1);
    b.vx1 = std::max(x0, x1);
    b.vy1 = std::max(y0, y1);
    b.marker_size = marker_size;
    b.cam = make_camera(K, D);
    b.dict = ctx->dict;
    return AB_OK;
}

// LINES refinement; the contour is undistorted first only with a distorted camera (cpp:957-959; all-zero coefficients
// make cv::undistortPoints the identity on pixel coordinates, see Camera::zero_D)
static void launch_refine_lines(const Batch& b, cudaStream_t st) {
    const dim3 grid(LINES_CTAS_PER_FRAME, b.B);
    if (b.cam.has_K && b.cam.has_D && !b.cam.zero_D) k_refine_lines<true><<<grid, 128, 0, st>>>(b);
    else k_refine_lines<false><<<grid, 128, 0, st>>>(b);
}

// k_trace<true>: every lane of the persistent grid owns a strip of max_len / 2 + 2 recorded pixel pairs (30 KB at 4K), so the
// grid is as large as the parked walks can use, WALKER_CTAS_PER_SM allows and the strip budget pays for.  Called once per
// batch, before its first launch.
static int plan_trace_long(ab_context* ctx, int max_len, unsigned cap_long) {
    const size_t half = ((size_t)(std::max(max_len, 0) / 2 + 2) + 1) & ~(size_t)1;  // even: 16-byte aligned strips
    size_t ctas = (size_t)ctx->sm_count * WALKER_CTAS_PER_SM;
    ctas = std::min(ctas, ((size_t)cap_long + 127) / 128);
    ctas = std::max<size_t>(1, std::min(ctas, ctx->trace_rec_budget / (half * 128 * sizeof(uint2))));
    const size_t need = ctas * 128 * half * sizeof(uint2);
    if (need > ctx->trace_rec_bytes) {  // grows only when the geometry or the maximum contour size grew
        if (ctx->d_trace_rec) cudaFree(ctx->d_trace_rec);
        ctx->d_trace_rec = nullptr;
        ctx->trace_rec_bytes = 0;
        cudaError_t e = cudaMalloc(&ctx->d_trace_rec, need);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return set_err(ctx, AB_E_CUDA, "walker strips (%zu MB): %s", need >> 20, cudaGetErrorString(e));
        }
        ctx->trace_rec_bytes = need;
    }
    ctx->rec_ctas = (unsigned)ctas;
    ctx->rec_half = (unsigned)half;
    return AB_OK;
}
static void launch_trace_long(ab_context* ctx, Batch& bv, cudaStream_t st) {
    bv.trace_rec = ctx->d_trace_rec;
    bv.rec_half = ctx->rec_half;
    k_trace<true><<<ctx->rec_ctas, 128, 0, st>>>(bv);
}

// board-stage buffers of this slot for the reserved geometry (maxB frames of capC markers)
static int ensure_board_buffers(ab_context* ctx) {
    if (ctx->board_frames >= ctx->maxB && ctx->board_capc == ctx->capC) return AB_OK;
    auto F = [](auto*& p) {
        if (p) cudaFree(p);
        p = nullptr;
    };
    F(ctx->d_boards);
    F(ctx->d_board_slots);
    F(ctx->d_board_pts);
    ctx->board_frames = ctx->board_capc = 0;
    const size_t B = (size_t)ctx->maxB, C = (size_t)ctx->capC;
    CK(cudaMalloc(&ctx->d_boards, B * sizeof(ab_board)));
    CK(cudaMalloc(&ctx->d_board_slots, B * C * sizeof(int32_t)));
    CK(cudaMalloc(&ctx->d_board_pts, B * C * BOARD_PTS_PER_MARKER * sizeof(float)));
    ctx->board_frames = ctx->maxB;
    ctx->board_capc = ctx->capC;
    return AB_OK;
}

// launches the whole path for frames resident at `dgrey`
static int run_batch(ab_context* ctx, const uint8_t* dgrey, size_t row, size_t frame, int n, const float* K,
                     const float* D, float marker_size) {
    const ab_params& P = ctx->params;
    if (P.decoder == AB_DECODER_HRM && !ctx->have_dict)
        return set_err(ctx, AB_E_STATE, "HRM decoder selected but no dictionary loaded (ab_load_hrm_dictionary)");
    if (P.decoder == AB_DECODER_HOST_CALLBACK && !ctx->cb)
        return set_err(ctx, AB_E_STATE, "host-callback decoder selected but no callback set");
    if (P.decoder == AB_DECODER_HRM && (ctx->dict.n + 2) > P.warp_size)
        return set_err(ctx, AB_E_INVALID, "warp size too small for the dictionary");
    if (P.corner_method == AB_CORNER_SUBPIX && ((int)P.thres_param1 < 1 || (int)P.thres_param1 > 24))
        return set_err(ctx, AB_E_INVALID, "SUBPIX window %d outside 1..24", (int)P.thres_param1);
    if (P.locked_corners && ((int)P.thres_param1 < 1 || (int)P.thres_param1 > 24))
        return set_err(ctx, AB_E_INVALID, "locked-corner window %d outside 1..24", (int)P.thres_param1);
    // setThresholdParamRange (markerdetector.h:152, cpp:322-334): 2*range+1 threshold images per frame, param1 =
    // p1 - range + range*i (sic, SURVEY B.6); they live as n_t consecutive "virtual frames" per frame for the
    // threshold / contour / polygon stages and are merged per frame by k_polygon's quad keys.
    // CANNY ignores the parameters: the reference's 2r+1 identical edge images yield duplicate candidates that its
    // too-near filter removes again (cpp:322-334, :592-627), so one image gives the same result.
    const int n_t = n_thres_images(P);
    if (n * n_t > ctx->maxB) return set_err(ctx, AB_E_STATE, "internal: %d virtual frames > reserved %d", n * n_t, ctx->maxB);
    {   // k_scan_starts indexes its work items with 32 bits
        const unsigned long long items = 8ull * (unsigned long long)((ctx->W + 31) >> 5) * (unsigned long long)((ctx->H + 2 + BIT_TILE - 1) / BIT_TILE) *
                                         (unsigned long long)(n * n_t);
        if (items >= (1ull << 32)) return set_err(ctx, AB_E_INVALID, "batch of %d frames %dx%d is too large for one launch: split it", n, ctx->W, ctx->H);
    }
    Batch b;
    fill_batch(ctx, b, dgrey, row, frame, n, n_t, K, D, marker_size);
    if (ctx->have_board) {
        if (int rc = ensure_board_buffers(ctx)) return rc;
        b.boards = ctx->d_boards;
        b.board_slots = ctx->d_board_slots;
        b.board_pts = ctx->d_board_pts;
    }
    cudaStream_t st = ctx->stream;
    const bool timing = ctx->timing;
    const int sms = ctx->sm_count;
    CK(cudaMemsetAsync(ctx->d_counters, 0, ctx->counters_bytes, st));
    if (int rc = plan_trace_long(ctx, b.max_len, b.cap_long)) return rc;
    if (timing) cudaEventRecord(ctx->ev[0], st);
    if (timing) cudaEventRecord(ctx->kev[0], st);
    for (int ti = 0; ti < n_t; ti++) {
        double p1 = n_t == 1 ? P.thres_param1 : P.thres_param1 - P.thres_param1_range + (double)P.thres_param1_range * ti;
        int rc = launch_threshold(ctx, b, P.thres_method, p1, P.thres_param2, n_t, ti, st);
        if (rc) return rc;
    }
    if (timing) cudaEventRecord(ctx->kev[1], st);
    Batch bv = b;  // the same buffers seen as n * n_t virtual frames
    bv.B = n * n_t;
    if (P.erosion) {
        k_erode<<<sms * 8, 256, 0, st>>>(bv.bits, bv.bits2, bv.thres, bv.bits_words, bv.W, bv.H, bv.wpr, bv.B);
        std::swap(bv.bits, bv.bits2);
        std::swap(b.bits, b.bits2);
    }
    if (timing) cudaEventRecord(ctx->ev[1], st);
    k_scan_starts<<<sms * 8, 256, 0, st>>>(bv);
    if (timing) cudaEventRecord(ctx->kev[2], st);
    k_trace<false><<<sms * WALKER_CTAS_PER_SM, 128, 0, st>>>(bv);
    if (timing) cudaEventRecord(ctx->kev[3], st);
    launch_trace_long(ctx, bv, st);
    if (timing) cudaEventRecord(ctx->kev[4], st);
    k_emit<<<sms * 8, 128, 0, st>>>(bv);
    if (timing) cudaEventRecord(ctx->kev[5], st);
    k_polygon<<<sms * 8, 128, 0, st>>>(bv);
    if (timing) cudaEventRecord(ctx->kev[6], st);
    k_frame_filter<<<n, 256, 0, st>>>(b);
    CK(cudaGetLastError());
    if (timing) cudaEventRecord(ctx->kev[7], st);
    if (timing) cudaEventRecord(ctx->ev[2], st);
    dim3 gcand(b.cap_c, n);
    dim3 gdec((b.cap_c + DECODE_WARPS - 1) / DECODE_WARPS, n);
    const size_t dec_smem = DECODE_WARPS * identify_smem_per_warp(b.S);
    if (dec_smem > 48 * 1024) cudaFuncSetAttribute(k_identify, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dec_smem);
    k_homography<<<dim3((b.cap_c + 63) / 64, n), 64, 0, st>>>(b);
    k_sample<<<gdec, 32 * DECODE_WARPS, 0, st>>>(b);
    if (timing) cudaEventRecord(ctx->kev[8], st);
    if (P.decoder == AB_DECODER_HOST_CALLBACK) {
        CK(cudaGetLastError());
        // MarkerdetectorFunc plugin hook (markerdetector.h:78,243): canonical images go to the host, the
        // user function runs per candidate in the reference's order, ids/rotations come back.
        std::vector<unsigned> ncand(n);
        CK(cudaMemcpyAsync(ncand.data(), b.n_cands, sizeof(unsigned) * n, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        size_t ss = (size_t)b.S * b.S;
        std::vector<uint8_t> canon((size_t)n * b.cap_c * ss);
        CK(cudaMemcpyAsync(canon.data(), b.canon, canon.size(), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        std::vector<int2> idrot((size_t)n * b.cap_c, make_int2(-1, 0));
        for (int f = 0; f < n; f++)
            for (unsigned c = 0; c < std::min<unsigned>(ncand[f], b.cap_c); c++) {
                int nrot = 0;
                int id = ctx->cb(canon.data() + ((size_t)f * b.cap_c + c) * ss, b.S, &nrot, ctx->cb_user);
                idrot[(size_t)f * b.cap_c + c] = make_int2(id, nrot);
            }
        DevBuf d_idrot;
        CK(d_idrot.alloc(idrot.size() * sizeof(int2)));
        CK(cudaMemcpyAsync(d_idrot.p, idrot.data(), idrot.size() * sizeof(int2), cudaMemcpyHostToDevice, st));
        k_set_ids<<<dim3((b.cap_c + 127) / 128, n), 128, 0, st>>>(b, d_idrot.as<int2>());
        CK(cudaStreamSynchronize(st));
    } else {
        k_otsu<<<dim3((b.cap_c + 31) / 32, n), 32, 0, st>>>(b);
        k_identify<<<gdec, 32 * DECODE_WARPS, dec_smem, st>>>(b);
        CK(cudaGetLastError());
    }
    if (timing) cudaEventRecord(ctx->kev[9], st);
    if (timing) cudaEventRecord(ctx->ev[3], st);
    if (P.locked_corners && (P.corner_method == AB_CORNER_HARRIS || P.corner_method == AB_CORNER_SUBPIX)) {
        // findCornerMaxima before the refiner (src/markerdetector.cpp:397-398)
        int w = b.subpix_win;
        size_t smem = (size_t)5 * (2 * w) * (2 * w) * sizeof(float);
        if (smem > 48 * 1024) cudaFuncSetAttribute(k_corner_maxima, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        k_corner_maxima<<<dim3(4 * b.cap_c, n), 64, smem, st>>>(b);
    }
    if (P.corner_method == AB_CORNER_LINES) {
        launch_refine_lines(b, st);
    } else if (P.corner_method == AB_CORNER_HARRIS) {
        k_refine_harris<<<dim3(b.cap_c, n), 128, 0, st>>>(b);
    } else if (P.corner_method == AB_CORNER_SUBPIX) {
        int w = b.subpix_win, pw = 2 * w + 3;
        size_t smem = (size_t)4 * pw * pw * sizeof(float);
        if (smem > 48 * 1024) cudaFuncSetAttribute(k_refine_subpix, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        k_refine_subpix<<<dim3(b.cap_c, n), 128, smem, st>>>(b);
    }
    CK(cudaGetLastError());
    if (timing) cudaEventRecord(ctx->kev[10], st);
    if (timing) cudaEventRecord(ctx->ev[4], st);
    k_finalize<<<n, 128, 0, st>>>(b);
    if (b.cam.has_K && b.marker_size > 0) k_pose<<<dim3((b.cap_c + 31) / 32, n), 32, 0, st>>>(b);
    CK(cudaGetLastError());
    if (timing) cudaEventRecord(ctx->kev[11], st);
    if (timing) cudaEventRecord(ctx->ev[5], st);
    if (b.boards) {
        k_board_batch<<<n, 32, 0, st>>>(b, ctx->board);
        CK(cudaGetLastError());
    }
    if (timing) cudaEventRecord(ctx->kev[12], st);
    ctx->last = b;
    ctx->have_last = true;
    ctx->last_n = n;
    return AB_OK;
}

static int check_device_errors(ab_context* ctx, const Counters* c) {
    if (!c->err) return AB_OK;
    std::string what;
    if (c->err & ERR_STARTS_OVERFLOW) what += " start-candidates(max_start_candidates_per_frame)";
    if (c->err & ERR_CONTOURS_OVERFLOW) what += " contours";
    if (c->err & ERR_POOL_OVERFLOW) what += " contour-points(max_contour_points_per_frame)";
    if (c->err & ERR_QUADS_OVERFLOW) what += " quads(max_quads_per_frame)";
    if (c->err & ERR_CANDS_OVERFLOW) what += " candidates(max_candidates_per_frame)";
    if (c->err & ERR_LINE_FIT) what += " line-fit-sweeps(LINES_MAX_SWEEPS)";
    return set_err(ctx, AB_E_CAPACITY, "device buffer overflow:%s -- results are incomplete; call ab_reserve with larger capacities",
                   what.c_str());
}

// the second set of per-batch buffers: a library-owned context that mirrors the owner's configuration
static int get_twin(ab_context* ctx, ab_context** out) {
    if (!ctx->twin) {
        ab_context* t = nullptr;
        int rc = ab_create(ctx->device, &t);
        if (rc) return set_err(ctx, rc, "cannot create the second in-flight context");
        t->owner = ctx;
        ctx->twin = t;
    }
    ab_context* t = ctx->twin;
    t->params = ctx->params;
    t->dict = ctx->dict;  // device pointers owned by `ctx`
    t->have_dict = ctx->have_dict;
    t->board = ctx->board;  // device arrays owned by `ctx`
    t->have_board = ctx->have_board;
    t->cb = ctx->cb;
    t->cb_user = ctx->cb_user;
    t->timing = ctx->timing;
    t->capLongPF = ctx->capLongPF;
    if (t->userQ != ctx->userQ || t->userC != ctx->userC || t->userStarts != ctx->userStarts || t->userPoints != ctx->userPoints) {
        free_buffers(t);
        t->userQ = ctx->userQ;
        t->userC = ctx->userC;
        t->userStarts = ctx->userStarts;
        t->userPoints = ctx->userPoints;
    }
    *out = t;
    return AB_OK;
}

static ab_context* slot_of(ab_context* ctx, int which) { return which ? ctx->twin : ctx; }
static ab_context* current_of(ab_context* ctx) { return (ctx->cur && ctx->twin) ? ctx->twin : ctx; }

// enqueue on this context or (when it still holds an un-fetched batch) on its twin
static int enqueue_on_free_slot(ab_context* ctx, const uint8_t* dev_frames, int width, int height, size_t row_stride,
                                size_t frame_stride, int n_frames, const float* K, const float* D, float marker_size) {
    if (ctx->n_pending >= 2)
        return set_err(ctx, AB_E_STATE, "two batches are already in flight: call ab_fetch_results before enqueueing a third");
    int which = ctx->n_pending == 1 ? 1 - ctx->pending[0] : 0;
    ab_context* tgt = ctx;
    if (which) {
        int rc = get_twin(ctx, &tgt);
        if (rc) return rc;
    }
    if (ctx->has_user_stream) {  // the frames were produced on the caller's stream
        CK(cudaEventRecord(ctx->ev_in, ctx->user_stream));
        CK(cudaStreamWaitEvent(tgt->stream, ctx->ev_in, 0));
    }
    int rc = ensure_reserved(tgt, width, height, n_frames * n_thres_images(ctx->params));
    if (rc) return rc;
    rc = run_batch(tgt, dev_frames, row_stride, frame_stride, n_frames, K, D, marker_size);
    if (rc) return rc;
    ctx->pending[ctx->n_pending++] = which;
    ctx->cur = which;
    return AB_OK;
}

int ab_enqueue_batch_device(ab_context* ctx, const uint8_t* dev_frames, int width, int height, size_t row_stride,
                            size_t frame_stride, int n_frames, const float* K, const float* D, float marker_size) {
    if (!ctx || !dev_frames || n_frames < 1 || row_stride < (size_t)width) return set_err(ctx, AB_E_INVALID, "bad arguments");
    cudaSetDevice(ctx->device);
    return enqueue_on_free_slot(ctx, dev_frames, width, height, row_stride, frame_stride, n_frames, K, D, marker_size);
}

// grow-only pinned host buffer
extern "C++" template <class T>
int ensure_pinned(ab_context* ctx, T*& p, size_t& have, size_t need) {
    if (need <= have) return AB_OK;
    if (p) cudaFreeHost(p);
    p = nullptr;
    have = 0;
    CK(cudaMallocHost(&p, need));
    have = need;
    return AB_OK;
}

// the owner's record of the boards of the batch being returned: cleared before its first chunk is fetched
static void reset_board_results(ab_context* ctx) {
    ctx->res_board = ctx->res_board_markers = true;
    ctx->res_boards.clear();
    ctx->res_markers.clear();
    ctx->res_off.assign(1, 0);
}

static int fetch_into(ab_context* ctx, ab_marker* out, int cap, int32_t* counts) {
    ab_context* own = ctx->owner ? ctx->owner : ctx;
    const bool board_ok = own->res_board;
    own->res_board = false;  // stays so when this fetch fails
    if (!ctx->have_last) return set_err(ctx, AB_E_STATE, "no batch has been run");
    const Batch& b = ctx->last;
    int n = ctx->last_n;
    cudaStream_t st = ctx->stream;
    int ncopy = std::min(cap, b.cap_c);
    if (int rc = ensure_pinned(ctx, ctx->h_markers, ctx->h_markers_bytes, (size_t)n * ncopy * sizeof(ab_marker))) return rc;
    CK(cudaMemcpyAsync(ctx->h_counters, ctx->d_counters, ctx->counters_bytes, cudaMemcpyDeviceToHost, st));
    if (out && ncopy > 0)
        CK(cudaMemcpy2DAsync(ctx->h_markers, (size_t)ncopy * sizeof(ab_marker), b.markers, (size_t)b.cap_c * sizeof(ab_marker),
                             (size_t)ncopy * sizeof(ab_marker), n, cudaMemcpyDeviceToHost, st));
    if (b.boards) {  // the board records and the matched slots (a frame's slots index its markers: < its count <= ncopy)
        if (int rc = ensure_pinned(ctx, ctx->h_boards, ctx->h_boards_bytes, (size_t)n * sizeof(ab_board))) return rc;
        CK(cudaMemcpyAsync(ctx->h_boards, b.boards, (size_t)n * sizeof(ab_board), cudaMemcpyDeviceToHost, st));
        if (out && ncopy > 0) {
            if (int rc = ensure_pinned(ctx, ctx->h_board_slots, ctx->h_board_slots_bytes, (size_t)n * ncopy * sizeof(int32_t))) return rc;
            CK(cudaMemcpy2DAsync(ctx->h_board_slots, (size_t)ncopy * sizeof(int32_t), b.board_slots, (size_t)b.cap_c * sizeof(int32_t),
                                 (size_t)ncopy * sizeof(int32_t), n, cudaMemcpyDeviceToHost, st));
        }
    }
    CK(cudaStreamSynchronize(st));
    int rc = check_device_errors(ctx, (const Counters*)ctx->h_counters);
    if (rc) return rc;
    const unsigned* nm = (const unsigned*)(ctx->h_counters + FRAME_COUNTS_OFFSET) + 2 * (size_t)ctx->maxB;
    for (int f = 0; f < n; f++) {
        if ((int)nm[f] > cap && out)
            return set_err(ctx, AB_E_CAPACITY, "frame %d has %u markers but cap_per_frame is %d", f, nm[f], cap);
        if (counts) counts[f] = (int32_t)nm[f];
        if (out) memcpy(out + (size_t)f * cap, ctx->h_markers + (size_t)f * ncopy, sizeof(ab_marker) * std::min<int>(nm[f], ncopy));
    }
    if (b.boards && board_ok) {
        for (int f = 0; f < n; f++) {
            const ab_board& bd = ctx->h_boards[f];
            own->res_boards.push_back(bd);
            for (int i = 0; out && i < bd.n_markers; i++) {
                ab_marker m = ctx->h_markers[(size_t)f * ncopy + ctx->h_board_slots[(size_t)f * ncopy + i]];
                m.ssize = bd.ssize;
                own->res_markers.push_back(m);
            }
            own->res_off.push_back((int32_t)own->res_markers.size());
        }
        own->res_board = true;
        own->res_board_markers = own->res_board_markers && out;
    }
    return AB_OK;
}

// results of the OLDEST un-fetched batch (enqueue order); with nothing pending: of the current batch again
static int fetch_oldest(ab_context* ctx, ab_marker* out, int cap, int32_t* counts) {
    int which = ctx->cur;
    if (ctx->n_pending) {
        which = ctx->pending[0];
        ctx->pending[0] = ctx->pending[1];
        ctx->n_pending--;
    }
    ctx->cur = which;
    reset_board_results(ctx);
    return fetch_into(slot_of(ctx, which), out, cap, counts);
}

int ab_fetch_results(ab_context* ctx, ab_marker* out, int cap_per_frame, int32_t* counts) {
    if (!ctx || cap_per_frame < 0) return AB_E_INVALID;
    cudaSetDevice(ctx->device);
    return fetch_oldest(ctx, out, cap_per_frame, counts);
}

static int ensure_grey(ab_context* ctx, size_t bytes) {
    if (ctx->grey_bytes >= bytes) return AB_OK;
    ctx->grey_bytes = 0;
    for (int i = 0; i < 2; i++) {
        if (ctx->d_grey[i]) cudaFree(ctx->d_grey[i]);
        ctx->d_grey[i] = nullptr;
    }
    for (int i = 0; i < 2; i++) CK(cudaMalloc(&ctx->d_grey[i], bytes));
    ctx->grey_bytes = bytes;
    return AB_OK;
}

// Host frames -> markers.  The batch goes through in chunks: the H2D copy of chunk c+1 (copy stream) runs under the
// kernels of chunk c, chunks alternate between this context and its twin so the kernels of chunk c+1 start under the
// latency-bound tail of chunk c, and the markers of chunk c-1 are copied back while chunk c runs.
static int detect_host(ab_context* ctx, const uint8_t* frames, int width, int height, size_t row_stride, size_t frame_stride,
                       int n_frames, const float* K, const float* D, float marker_size, ab_marker* out, int cap, int32_t* counts,
                       int channels) {
    if (!ctx || !frames || n_frames < 1 || row_stride < (size_t)width * channels || cap < 0)
        return set_err(ctx, AB_E_INVALID, "bad arguments");
    if (ctx->n_pending) return set_err(ctx, AB_E_STATE, "%d enqueued batch(es) not fetched yet", ctx->n_pending);
    cudaSetDevice(ctx->device);
    reset_board_results(ctx);
    // chunk size: what was reserved for this geometry, else up to 32 frames
    const int n_t = n_thres_images(ctx->params);
    int chunk = (ctx->W == width && ctx->H == height && ctx->maxB >= n_t) ? std::min(ctx->maxB / n_t, n_frames) : std::min(n_frames, 32);
    int rc = ensure_reserved(ctx, width, height, chunk * n_t);
    if (rc) return rc;
    chunk = std::min(ctx->maxB / n_t, n_frames);
    const size_t fpx = (size_t)width * height;
    const int nchunks = (n_frames + chunk - 1) / chunk;
    const bool two = nchunks > 1 && channels == 1 && ctx->params.decoder != AB_DECODER_HOST_CALLBACK;
    ab_context* slot[2] = {ctx, ctx};
    if (two) {
        rc = get_twin(ctx, &slot[1]);
        if (rc) return rc;
        rc = ensure_reserved(slot[1], width, height, chunk * n_t);
        if (rc) return rc;
        rc = ensure_grey(slot[1], fpx * chunk);
        if (rc) return rc;
    }
    rc = ensure_grey(ctx, fpx * chunk);
    if (rc) return rc;
    if (channels == 3 && ctx->bgr_bytes < fpx * 3 * chunk) {
        if (ctx->d_bgr) cudaFree(ctx->d_bgr);
        ctx->d_bgr = nullptr;
        ctx->bgr_bytes = 0;
        CK(cudaMalloc(&ctx->d_bgr, fpx * 3 * chunk));
        ctx->bgr_bytes = fpx * 3 * chunk;
    }
    auto staging = [&](int c) -> uint8_t* { return two ? slot[c & 1]->d_grey[0] : ctx->d_grey[c & 1]; };
    auto upload = [&](int c) -> int {
        int f0 = c * chunk, nf = std::min(chunk, n_frames - f0);
        int buf = c & 1;
        if (c >= 2) CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_done[buf], 0));  // chunk c-2 has read this buffer
        uint8_t* dst = staging(c);
        if (channels == 1) {
            if (frame_stride == row_stride * (size_t)height) {
                CK(cudaMemcpy2DAsync(dst, width, frames + (size_t)f0 * frame_stride, row_stride, width, (size_t)height * nf,
                                     cudaMemcpyHostToDevice, ctx->copy_stream));
            } else {
                for (int f = 0; f < nf; f++)
                    CK(cudaMemcpy2DAsync(dst + (size_t)f * fpx, width, frames + (size_t)(f0 + f) * frame_stride, row_stride, width,
                                         height, cudaMemcpyHostToDevice, ctx->copy_stream));
            }
        } else {
            for (int f = 0; f < nf; f++)
                CK(cudaMemcpy2DAsync(ctx->d_bgr + (size_t)f * fpx * 3, (size_t)width * 3, frames + (size_t)(f0 + f) * frame_stride,
                                     row_stride, (size_t)width * 3, height, cudaMemcpyHostToDevice, ctx->copy_stream));
            const size_t groups = (size_t)((width + 3) / 4) * height * nf;
            const int blocks = (int)std::min<size_t>((groups + 255) / 256, (size_t)ctx->sm_count * 16);
            k_bgr2grey<<<blocks, 256, 0, ctx->copy_stream>>>(ctx->d_bgr, (size_t)width * 3, fpx * 3, dst, width, height, nf);
        }
        CK(cudaEventRecord(ctx->ev_h2d[buf], ctx->copy_stream));
        return AB_OK;
    };
    auto fetch_chunk = [&](int c) -> int {
        const int f0 = c * chunk;
        return fetch_into(two ? slot[c & 1] : ctx, out ? out + (size_t)f0 * cap : nullptr, cap, counts ? counts + f0 : nullptr);
    };
    rc = upload(0);
    if (rc) return rc;
    for (int c = 0; c < nchunks; c++) {
        const int f0 = c * chunk, nf = std::min(chunk, n_frames - f0);
        const int buf = c & 1;
        ab_context* tgt = two ? slot[buf] : ctx;
        if (c + 1 < nchunks && channels == 1) {
            rc = upload(c + 1);
            if (rc) return rc;
        }
        CK(cudaStreamWaitEvent(tgt->stream, ctx->ev_h2d[buf], 0));
        rc = run_batch(tgt, staging(c), width, fpx, nf, K, D, marker_size);
        if (rc) return rc;
        CK(cudaEventRecord(ctx->ev_done[buf], tgt->stream));
        if (two) {
            if (c >= 1) {
                rc = fetch_chunk(c - 1);
                if (rc) return rc;
            }
        } else {
            rc = fetch_chunk(c);
            if (rc) return rc;
            if (c + 1 < nchunks && channels == 3) {  // the BGR staging buffer is single: upload after the fetch
                rc = upload(c + 1);
                if (rc) return rc;
            }
        }
    }
    if (two) {
        rc = fetch_chunk(nchunks - 1);
        if (rc) return rc;
    }
    ctx->cur = two ? ((nchunks - 1) & 1) : 0;  // the state getters read the last chunk
    return AB_OK;
}

int ab_detect_batch(ab_context* ctx, const uint8_t* frames, int width, int height, size_t row_stride, size_t frame_stride,
                    int n_frames, const float* K, const float* D, float marker_size, ab_marker* out, int cap_per_frame,
                    int32_t* counts) {
    return detect_host(ctx, frames, width, height, row_stride, frame_stride, n_frames, K, D, marker_size, out, cap_per_frame,
                       counts, 1);
}

int ab_detect_batch_bgr(ab_context* ctx, const uint8_t* frames, int width, int height, size_t row_stride, size_t frame_stride,
                        int n_frames, const float* K, const float* D, float marker_size, ab_marker* out, int cap_per_frame,
                        int32_t* counts) {
    return detect_host(ctx, frames, width, height, row_stride, frame_stride, n_frames, K, D, marker_size, out, cap_per_frame,
                       counts, 3);
}

// ---- state of the last batch ---------------------------------------------------------------------------
int ab_get_thresholded(ab_context* ctx, int frame, uint8_t* dst, size_t dst_stride) {
    if (ctx) ctx = current_of(ctx);
    if (!ctx || !ctx->have_last || frame < 0 || frame >= ctx->last_n || !dst) return set_err(ctx, AB_E_INVALID, "bad frame");
    cudaSetDevice(ctx->device);
    const Batch& b = ctx->last;
    // `thres` = the middle threshold image (thres_images[n_param1 / 2], markerdetector.cpp:334)
    CK(cudaMemcpy2DAsync(dst, dst_stride, b.thres + ((size_t)frame * b.n_t + b.n_t / 2) * b.W * b.H, b.W, b.W, b.H,
                         cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return AB_OK;
}

int ab_get_grey(ab_context* ctx, int frame, uint8_t* dst, size_t dst_stride) {
    if (ctx) ctx = current_of(ctx);
    if (!ctx || !ctx->have_last || frame < 0 || frame >= ctx->last_n || !dst) return set_err(ctx, AB_E_INVALID, "bad frame");
    cudaSetDevice(ctx->device);
    const Batch& b = ctx->last;
    CK(cudaMemcpy2DAsync(dst, dst_stride, b.grey + (size_t)frame * b.grey_frame, b.grey_row, b.W, b.H, cudaMemcpyDeviceToHost,
                         ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return AB_OK;
}

int ab_get_candidates(ab_context* ctx, int frame, float* quads, int32_t* ids, int32_t* n_rot, int cap, int32_t* n) {
    if (ctx) ctx = current_of(ctx);
    if (!ctx || !ctx->have_last || frame < 0 || frame >= ctx->last_n || !n) return set_err(ctx, AB_E_INVALID, "bad frame");
    cudaSetDevice(ctx->device);
    const Batch& b = ctx->last;
    CK(cudaStreamSynchronize(ctx->stream));
    unsigned nc = 0;
    CK(cudaMemcpy(&nc, b.n_cands + frame, sizeof(unsigned), cudaMemcpyDeviceToHost));
    nc = std::min<unsigned>(nc, b.cap_c);
    *n = (int32_t)nc;
    if ((int)nc > cap) return set_err(ctx, AB_E_CAPACITY, "%u candidates > cap %d", nc, cap);
    std::vector<CandRec> h(nc);
    if (nc) CK(cudaMemcpy(h.data(), b.cands + (size_t)frame * b.cap_c, sizeof(CandRec) * nc, cudaMemcpyDeviceToHost));
    for (unsigned i = 0; i < nc; i++) {
        if (quads) memcpy(quads + 8 * i, h[i].c, sizeof(float) * 8);
        if (ids) ids[i] = h[i].id;
        if (n_rot) n_rot[i] = h[i].nrot;
    }
    return AB_OK;
}

int ab_get_canonical(ab_context* ctx, int frame, int candidate, uint8_t* dst) {
    if (ctx) ctx = current_of(ctx);
    if (!ctx || !ctx->have_last || frame < 0 || frame >= ctx->last_n || !dst || candidate < 0 || candidate >= ctx->last.cap_c)
        return set_err(ctx, AB_E_INVALID, "bad frame/candidate");
    cudaSetDevice(ctx->device);
    const Batch& b = ctx->last;
    CK(cudaStreamSynchronize(ctx->stream));
    size_t ss = (size_t)b.S * b.S;
    CK(cudaMemcpy(dst, b.canon + ((size_t)frame * b.cap_c + candidate) * ss, ss, cudaMemcpyDeviceToHost));
    return AB_OK;
}

int ab_get_canonical_size(ab_context* ctx, int32_t* size) {
    if (ctx) ctx = current_of(ctx);
    if (!ctx || !ctx->have_last || !size) return set_err(ctx, AB_E_STATE, "no batch");
    *size = ctx->last.S;
    return AB_OK;
}

int ab_get_contour(ab_context* ctx, int frame, int candidate, int32_t* xy, int cap_points, int32_t* n) {
    if (ctx) ctx = current_of(ctx);
    if (!ctx || !ctx->have_last || frame < 0 || frame >= ctx->last_n || !n || candidate < 0 || candidate >= ctx->last.cap_c)
        return set_err(ctx, AB_E_INVALID, "bad frame/candidate");
    cudaSetDevice(ctx->device);
    const Batch& b = ctx->last;
    CK(cudaStreamSynchronize(ctx->stream));
    CandRec cr;
    CK(cudaMemcpy(&cr, b.cands + (size_t)frame * b.cap_c + candidate, sizeof(CandRec), cudaMemcpyDeviceToHost));
    // contour indices and point offsets are relative to the start of the batch's lists
    ContourRec rec;
    CK(cudaMemcpy(&rec, b.contours + cr.contour, sizeof(ContourRec), cudaMemcpyDeviceToHost));
    *n = (int32_t)rec.n;
    if ((int)rec.n > cap_points) return set_err(ctx, AB_E_CAPACITY, "contour has %u points > cap %d", rec.n, cap_points);
    std::vector<uint32_t> p(rec.n);
    CK(cudaMemcpy(p.data(), b.pool + rec.off, sizeof(uint32_t) * rec.n, cudaMemcpyDeviceToHost));
    for (uint32_t i = 0; i < rec.n; i++) {
        uint32_t v = cr.swapped ? p[rec.n - 1 - i] : p[i];  // the reference reverses swapped contours (:622-625)
        xy[2 * i] = (int32_t)(v & 0xFFFFu);
        xy[2 * i + 1] = (int32_t)(v >> 16);
    }
    return AB_OK;
}

int ab_get_counters(ab_context* ctx, int64_t* counters, int n) {
    if (ctx) ctx = current_of(ctx);
    if (!ctx || !ctx->have_last || !counters) return set_err(ctx, AB_E_INVALID, "no batch");
    cudaSetDevice(ctx->device);
    CK(cudaStreamSynchronize(ctx->stream));
    Counters c;
    CK(cudaMemcpy(&c, ctx->d_counters, sizeof(c), cudaMemcpyDeviceToHost));
    const int64_t v[6] = {(int64_t)c.n_starts,      (int64_t)c.n_contours,    (int64_t)c.pool_used,
                          (int64_t)c.n_quads_total, (int64_t)c.n_cands_total, (int64_t)c.n_markers_total};
    for (int i = 0; i < n && i < 6; i++) counters[i] = v[i];
    return AB_OK;
}

int ab_get_stage_ms(ab_context* ctx, float* ms, int n) {
    if (ctx) ctx = current_of(ctx);
    if (!ctx || !ms || !ctx->timing || !ctx->have_last) return set_err(ctx, AB_E_STATE, "timing not enabled");
    cudaSetDevice(ctx->device);
    CK(cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < n && i < 5; i++) CK(cudaEventElapsedTime(&ms[i], ctx->ev[i], ctx->ev[i + 1]));
    return AB_OK;
}

int ab_get_kernel_ms(ab_context* ctx, float* ms, int n) {
    if (ctx) ctx = current_of(ctx);
    if (!ctx || !ms || !ctx->timing || !ctx->have_last) return set_err(ctx, AB_E_STATE, "timing not enabled");
    cudaSetDevice(ctx->device);
    CK(cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < n && i < 12; i++) CK(cudaEventElapsedTime(&ms[i], ctx->kev[i], ctx->kev[i + 1]));
    return AB_OK;
}

// ---- public workers ---------------------------------------------------------------------------------------
int ab_threshold(ab_context* ctx, const uint8_t* grey, int width, int height, size_t row_stride, int method, double param1,
                 double param2, uint8_t* out, size_t out_stride) {
    if (!ctx || !grey || !out) return AB_E_INVALID;
    if (ctx->n_pending) return set_err(ctx, AB_E_STATE, "%d enqueued batch(es) not fetched yet", ctx->n_pending);
    ctx->cur = 0;
    cudaSetDevice(ctx->device);
    int rc = ensure_reserved(ctx, width, height, 1);
    if (rc) return rc;
    rc = ensure_grey(ctx, (size_t)width * height);
    if (rc) return rc;
    // markerdetector.cpp:646-649: -1 selects the stored parameters
    if (param1 == -1) param1 = ctx->params.thres_param1;
    if (param2 == -1) param2 = ctx->params.thres_param2;
    CK(cudaMemcpy2DAsync(ctx->d_grey[0], width, grey, row_stride, width, height, cudaMemcpyHostToDevice, ctx->stream));
    Batch b;
    fill_batch(ctx, b, ctx->d_grey[0], width, (size_t)width * height, 1, 1, nullptr, nullptr, -1.f);
    ctx->worker_call = true;
    rc = launch_threshold(ctx, b, method, param1, param2);
    ctx->worker_call = false;
    if (rc) return rc;
    CK(cudaMemcpy2DAsync(out, out_stride, b.thres, width, width, height, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return AB_OK;
}

int ab_detect_rectangles(ab_context* ctx, const uint8_t* thres, int width, int height, size_t row_stride, float* quads, int cap,
                         int32_t* n) {
    if (!ctx || !thres || !n) return AB_E_INVALID;
    if (ctx->n_pending) return set_err(ctx, AB_E_STATE, "%d enqueued batch(es) not fetched yet", ctx->n_pending);
    ctx->cur = 0;
    cudaSetDevice(ctx->device);
    int rc = ensure_reserved(ctx, width, height, 1);
    if (rc) return rc;
    rc = ensure_grey(ctx, (size_t)width * height);
    if (rc) return rc;
    cudaStream_t st = ctx->stream;
    CK(cudaMemcpy2DAsync(ctx->d_grey[0], width, thres, row_stride, width, height, cudaMemcpyHostToDevice, st));
    Batch b;
    fill_batch(ctx, b, ctx->d_grey[0], width, (size_t)width * height, 1, 1, nullptr, nullptr, -1.f);
    CK(cudaMemsetAsync(ctx->d_counters, 0, ctx->counters_bytes, st));
    k_threshold_fixed<<<ctx->sm_count * 8, 256, 0, st>>>(b.grey, b.grey_row, b.grey_frame, b.thres, b.bits, b.bits_words, b.W, b.H,
                                                          b.wpr, 0, 1, 1, 1, 0);
    k_scan_starts<<<ctx->sm_count * 8, 256, 0, st>>>(b);
    k_trace<false><<<ctx->sm_count * WALKER_CTAS_PER_SM, 128, 0, st>>>(b);
    rc = plan_trace_long(ctx, b.max_len, b.cap_long);
    if (rc) return rc;
    launch_trace_long(ctx, b, st);
    k_emit<<<ctx->sm_count * 8, 128, 0, st>>>(b);
    k_polygon<<<ctx->sm_count * 4, 128, 0, st>>>(b);
    k_frame_filter<<<1, 256, 0, st>>>(b);
    CK(cudaGetLastError());
    ctx->last = b;
    ctx->have_last = true;
    ctx->last_n = 1;
    CK(cudaMemcpyAsync(ctx->h_counters, ctx->d_counters, ctx->counters_bytes, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    rc = check_device_errors(ctx, (const Counters*)ctx->h_counters);
    if (rc) return rc;
    return ab_get_candidates(ctx, 0, quads, nullptr, nullptr, cap, n);
}

int ab_warp(ab_context* ctx, const uint8_t* grey, int width, int height, size_t row_stride, const float* quad, int size,
            uint8_t* out) {
    if (!ctx || !grey || !quad || !out || size < 1 || size > 1024 || width < 1 || height < 1 || row_stride < (size_t)width)
        return set_err(ctx, AB_E_INVALID, "bad arguments");
    cudaSetDevice(ctx->device);
    cudaStream_t st = ctx->stream;
    DevBuf d_img, d_out, d_quad;
    CK(d_img.alloc((size_t)width * height));
    CK(d_out.alloc((size_t)size * size));
    CK(d_quad.alloc(8 * sizeof(float)));
    CK(cudaMemcpy2DAsync(d_img.p, width, grey, row_stride, width, height, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_quad.p, quad, 8 * sizeof(float), cudaMemcpyHostToDevice, st));
    k_warp_single<<<1, 256, 0, st>>>(d_img.as<uint8_t>(), width, height, width, d_quad.as<float>(), size, d_out.as<uint8_t>());
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, d_out.p, (size_t)size * size, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return AB_OK;
}

// MarkerDetector::refineCandidateLines (h:280, cpp:931-997) for one candidate
int ab_refine_candidate_lines(ab_context* ctx, const int32_t* contour_xy, int n_points, float* corners, const float* K,
                              const float* D) {
    if (!ctx || !contour_xy || !corners || n_points < 4 || n_points > (1 << 24))
        return set_err(ctx, AB_E_INVALID, "refineCandidateLines: bad arguments");
    std::vector<uint32_t> packed((size_t)n_points);
    for (int i = 0; i < n_points; i++) {
        const int32_t x = contour_xy[2 * i], y = contour_xy[2 * i + 1];
        if (x < 0 || y < 0 || x > 0xFFFF || y > 0xFFFF) return set_err(ctx, AB_E_INVALID, "refineCandidateLines: contour point outside 0..65535");
        packed[i] = (uint32_t)x | ((uint32_t)y << 16);
    }
    cudaSetDevice(ctx->device);
    cudaStream_t st = ctx->stream;
    DevBuf d_pts, d_io, d_err;
    CK(d_pts.alloc(packed.size() * 4));
    CK(d_io.alloc(16 * sizeof(float)));
    CK(d_err.alloc(sizeof(unsigned)));
    CK(cudaMemcpyAsync(d_pts.p, packed.data(), packed.size() * 4, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_io.p, corners, 8 * sizeof(float), cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(d_io.as<float>() + 8, 0xFF, 8 * sizeof(float), st));  // NaN pattern: "corner not found on the contour"
    CK(cudaMemsetAsync(d_err.p, 0, sizeof(unsigned), st));
    // the reference undistorts only when both matrices are given (cpp:957-959)
    const Camera cam = make_camera(K && D ? K : nullptr, K && D ? D : nullptr);
    if (cam.has_K && cam.has_D && !cam.zero_D)
        k_refine_lines_single<true><<<1, 128, 0, st>>>(d_pts.as<uint32_t>(), n_points, d_io.as<float>(), cam, d_io.as<float>() + 8, d_err.as<unsigned>());
    else
        k_refine_lines_single<false><<<1, 128, 0, st>>>(d_pts.as<uint32_t>(), n_points, d_io.as<float>(), cam, d_io.as<float>() + 8, d_err.as<unsigned>());
    CK(cudaGetLastError());
    float res[8];
    unsigned err = 0;
    CK(cudaMemcpyAsync(res, d_io.as<float>() + 8, sizeof(res), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&err, d_err.p, sizeof(err), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (err) return set_err(ctx, AB_E_CAPACITY, "refineCandidateLines: line fit did not converge within the sweeps the kernel replays");
    if (res[0] != res[0]) return set_err(ctx, AB_E_INVALID, "refineCandidateLines: a corner is not a point of the contour");
    memcpy(corners, res, sizeof(res));
    return AB_OK;
}

// ---- marker / board rendering (k_render.cuh) -----------------------------------------------------------------
static int render_canvas(ab_context* ctx, int W, int H, uint8_t background, const std::vector<RenderRect>& rects, int n_black,
                         uint8_t* out, size_t out_stride) {
    cudaSetDevice(ctx->device);
    DevBuf d_img, d_rects;
    CK(d_img.alloc((size_t)W * H));
    k_fill_u8<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(d_img.as<uint8_t>(), (size_t)W * H, background);
    if (!rects.empty()) {
        CK(d_rects.alloc(rects.size() * sizeof(RenderRect)));
        CK(cudaMemcpyAsync(d_rects.p, rects.data(), rects.size() * sizeof(RenderRect), cudaMemcpyHostToDevice, ctx->stream));
        int maxs = 1;
        for (const auto& r : rects) maxs = std::max(maxs, r.size);
        dim3 grid((unsigned)std::min(1024, (maxs * maxs + 255) / 256), (unsigned)rects.size());
        k_render_fiducidal<<<grid, 256, 0, ctx->stream>>>(d_img.as<uint8_t>(), W, H, d_rects.as<RenderRect>(), n_black);
    }
    CK(cudaGetLastError());
    CK(cudaMemcpy2DAsync(out, out_stride, d_img.p, W, W, H, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return AB_OK;
}

int ab_create_marker_image(ab_context* ctx, int id, int size, int locked, uint8_t* out, size_t out_stride, int* out_side) {
    if (!ctx) return AB_E_INVALID;
    if (id < 0 || id >= 1024) return set_err(ctx, AB_E_INVALID, "createMarkerImage: 0 <= id < 1024");  // CV_Assert, cpp:214
    if (size < 1 || size > 16384) return set_err(ctx, AB_E_INVALID, "createMarkerImage: bad size");
    const int sq = locked ? (int)((float)size * 0.25f) : 0;  // cpp:241
    const int side = size + 2 * sq;
    if (out_side) *out_side = side;
    if (!out) return AB_OK;
    if (out_stride < (size_t)side) return set_err(ctx, AB_E_INVALID, "createMarkerImage: stride too small");
    std::vector<RenderRect> rects;
    if (locked) {  // four black squares in the corners of a white canvas (cpp:243-254)
        rects.push_back(RenderRect{0, 0, sq, 0});
        rects.push_back(RenderRect{0, side - sq, sq, 0});
        rects.push_back(RenderRect{side - sq, side - sq, sq, 0});
        rects.push_back(RenderRect{side - sq, 0, sq, 0});
    }
    const int n_black = (int)rects.size();
    rects.push_back(RenderRect{sq, sq, size, id});
    return render_canvas(ctx, side, side, locked ? 255 : 0, rects, n_black, out, out_stride);
}

int ab_create_board_image(ab_context* ctx, int kind, int grid_w, int grid_h, int marker_size, int marker_distance, int center_data,
                          const int32_t* ids, int n_ids, uint8_t* out, size_t out_stride, int* out_w, int* out_h, int32_t* ids_out,
                          float* corners_out, int cap, int* n_out) {
    if (!ctx) return AB_E_INVALID;
    if (kind < 0 || kind > 2 || grid_w < 1 || grid_h < 1 || marker_size < 7 || marker_distance < 0 || (long long)grid_w * grid_h > 65536)
        return set_err(ctx, AB_E_INVALID, "createBoardImage: bad arguments");
    const int dist = kind == 1 ? 0 : marker_distance;  // the chessboard has no gaps
    const int step = marker_size + dist;
    const int sizeY = grid_h * marker_size + (grid_h - 1) * dist, sizeX = grid_w * marker_size + (grid_w - 1) * dist;
    const int centerX = sizeX / 2, centerY = sizeY / 2;
    if ((long long)sizeX * sizeY > (1ll << 30)) return set_err(ctx, AB_E_INVALID, "createBoardImage: image too large");
    std::vector<RenderRect> rects;
    for (int y = 0; y < grid_h; y++) {
        bool toWrite = (y % 2) != 0;  // chessboard: alternate, starting with a marker on even rows (cpp:355-361)
        for (int x = 0; x < grid_w; x++) {
            toWrite = !toWrite;
            const bool use = kind == 0 ? true : (kind == 1 ? toWrite : (y == 0 || y == grid_h - 1 || x == 0 || x == grid_w - 1));
            if (use) rects.push_back(RenderRect{x * step, y * step, marker_size, 0});
        }
    }
    const int n = (int)rects.size();
    if (out_w) *out_w = sizeX;
    if (out_h) *out_h = sizeY;
    if (n_out) *n_out = n;
    if (!out) return AB_OK;
    if (!ids || n_ids < n) return set_err(ctx, AB_E_INVALID, "createBoardImage: %d marker ids needed", n);
    if (cap < n || !ids_out || !corners_out) return set_err(ctx, AB_E_CAPACITY, "createBoardImage: room for %d markers needed", n);
    if (out_stride < (size_t)sizeX) return set_err(ctx, AB_E_INVALID, "createBoardImage: stride too small");
    const bool center = kind == 0 ? true : center_data != 0;
    for (int i = 0; i < n; i++) {
        if (ids[i] < 0 || ids[i] >= 1024) return set_err(ctx, AB_E_INVALID, "createBoardImage: 0 <= id < 1024");
        rects[i].id = ids[i];
        ids_out[i] = ids[i];
        const float x0 = (float)rects[i].x0, y0 = (float)rects[i].y0, s = (float)marker_size;
        const float c[12] = {x0, y0, 0, x0 + s, y0, 0, x0 + s, y0 + s, 0, x0, y0 + s, 0};
        for (int k = 0; k < 4; k++) {
            corners_out[12 * i + 3 * k] = c[3 * k] - (center ? (float)centerX : 0.f);
            corners_out[12 * i + 3 * k + 1] = c[3 * k + 1] - (center ? (float)centerY : 0.f);
            corners_out[12 * i + 3 * k + 2] = 0.f;
        }
    }
    return render_canvas(ctx, sizeX, sizeY, 255, rects, 0, out, out_stride);
}

int ab_create_hrm_marker_image(ab_context* ctx, int n, const uint8_t* bits, int pix_size, uint8_t* out, size_t out_stride, int* out_side) {
    if (!ctx) return AB_E_INVALID;
    if (n < 1 || n > 8 || pix_size < 1 || pix_size > 16384) return set_err(ctx, AB_E_INVALID, "getImg: bad arguments");
    const int nrows = n + 2;
    if (pix_size % nrows != 0) pix_size = pix_size + nrows - pix_size % nrows;  // hrm.cpp:237-238
    if (out_side) *out_side = pix_size;
    if (!out) return AB_OK;
    if (!bits || out_stride < (size_t)pix_size) return set_err(ctx, AB_E_INVALID, "getImg: bad arguments");
    cudaSetDevice(ctx->device);
    DevBuf d_img, d_bits;
    CK(d_img.alloc((size_t)pix_size * pix_size));
    CK(d_bits.alloc((size_t)n * n));
    CK(cudaMemcpyAsync(d_bits.p, bits, (size_t)n * n, cudaMemcpyHostToDevice, ctx->stream));
    k_render_hrm<<<std::min(1024, (pix_size * pix_size + 255) / 256), 256, 0, ctx->stream>>>(d_img.as<uint8_t>(), pix_size, n,
                                                                                             d_bits.as<uint8_t>());
    CK(cudaGetLastError());
    CK(cudaMemcpy2DAsync(out, out_stride, d_img.p, pix_size, pix_size, pix_size, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return AB_OK;
}

int ab_create_hrm_board_image(ab_context* ctx, int grid_w, int grid_h, int n, const uint8_t* bits, int count, uint8_t* out,
                              size_t out_stride, int* out_w, int* out_h, int32_t* ids_out, float* corners_out, int cap, int* n_out) {
    if (!ctx) return AB_E_INVALID;
    if (grid_w < 1 || grid_h < 1 || n < 1 || n > 8 || (long long)grid_w * grid_h > 65536) return set_err(ctx, AB_E_INVALID, "createBoardImage: bad arguments");
    const int ms = (n + 2) * 20, md = ms / 5;  // hrm.cpp:500-501
    const int sizeY = grid_h * ms + (grid_h - 1) * md, sizeX = grid_w * ms + (grid_w - 1) * md;
    const float centerX = (float)(sizeX / 2.), centerY = (float)(sizeY / 2.);
    const int nm = grid_w * grid_h;
    if (out_w) *out_w = sizeX;
    if (out_h) *out_h = sizeY;
    if (n_out) *n_out = nm;
    if (!out) return AB_OK;
    if (!bits || count < nm) return set_err(ctx, AB_E_INVALID, "createBoardImage: the dictionary has %d markers, %d needed", count, nm);
    if (cap < nm || !ids_out || !corners_out) return set_err(ctx, AB_E_CAPACITY, "createBoardImage: room for %d markers needed", nm);
    if (out_stride < (size_t)sizeX) return set_err(ctx, AB_E_INVALID, "createBoardImage: stride too small");
    std::vector<RenderRect> rects;
    int idp = 0;
    for (int y = 0; y < grid_h; y++)
        for (int x = 0; x < grid_w; x++, idp++) {
            rects.push_back(RenderRect{x * (md + ms), y * (md + ms), ms, idp});
            uint8_t code[64];
            for (int i = 0; i < n * n; i++) code[i] = bits[(size_t)idp * n * n + i] != 0;
            uint64_t rb[4];
            uint32_t rid[4];
            hrm_rotations(code, n, rb, rid);
            ids_out[idp] = (int32_t)rid[0];  // MarkerCode::getId()
            const float x0 = (float)(x * (md + ms)) - centerX, y0 = (float)(y * (md + ms)) - centerY, s = (float)ms;
            // y negated so that the z axis points up (hrm.cpp:536-540)
            const float c[12] = {x0, -y0, 0, x0 + s, -y0, 0, x0 + s, -(y0 + s), 0, x0, -(y0 + s), 0};
            for (int k = 0; k < 12; k++) corners_out[12 * idp + k] = c[k];
        }
    cudaSetDevice(ctx->device);
    DevBuf d_img, d_bits, d_rects;
    CK(d_img.alloc((size_t)sizeX * sizeY));
    CK(d_bits.alloc((size_t)nm * n * n));
    CK(d_rects.alloc(rects.size() * sizeof(RenderRect)));
    CK(cudaMemcpyAsync(d_bits.p, bits, (size_t)nm * n * n, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_rects.p, rects.data(), rects.size() * sizeof(RenderRect), cudaMemcpyHostToDevice, ctx->stream));
    k_fill_u8<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(d_img.as<uint8_t>(), (size_t)sizeX * sizeY, 255);
    k_render_hrm_board<<<dim3((unsigned)((ms * ms + 255) / 256), (unsigned)nm), 256, 0, ctx->stream>>>(
        d_img.as<uint8_t>(), sizeX, sizeY, d_rects.as<RenderRect>(), n, d_bits.as<uint8_t>());
    CK(cudaGetLastError());
    CK(cudaMemcpy2DAsync(out, out_stride, d_img.p, sizeX, sizeX, sizeY, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return AB_OK;
}

int ab_calculate_extrinsics(ab_context* ctx, ab_marker* markers, int n, const float* K, const float* D, float marker_size,
                            int set_y_perp) {
    if (!ctx || !markers || n < 0 || !K || !(marker_size > 0)) return set_err(ctx, AB_E_INVALID, "calculateExtrinsics: invalid arguments");
    if (n == 0) return AB_OK;
    cudaSetDevice(ctx->device);
    DevBuf d;
    CK(d.alloc(sizeof(ab_marker) * n));
    CK(cudaMemcpyAsync(d.p, markers, sizeof(ab_marker) * n, cudaMemcpyHostToDevice, ctx->stream));
    k_extrinsics<<<(n + 63) / 64, 64, 0, ctx->stream>>>(d.as<ab_marker>(), n, make_camera(K, D), marker_size, set_y_perp);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(markers, d.p, sizeof(ab_marker) * n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return AB_OK;
}

// BoardDetector::detect's constants of a configuration (boarddetector.cpp:95-136), computed once on the host: the kernel
// must not recompute d01 (a contracted sum of products would change its bits)
static BoardArgs board_args(const ab_board_config* cfg, const float* K, const float* D, float marker_size, float repj_err_thres,
                            int set_y_perp) {
    BoardArgs a;
    memset(&a, 0, sizeof(a));
    const float* c0 = cfg->corners;
    double d01 = sqrt((double)(c0[0] - c0[3]) * (c0[0] - c0[3]) + (double)(c0[1] - c0[4]) * (c0[1] - c0[4]) + (double)(c0[2] - c0[5]) * (c0[2] - c0[5]));
    a.ssize = -1.f;
    if (cfg->info_type == 0 && marker_size > 0) a.ssize = marker_size;
    else if (cfg->info_type == 1) a.ssize = (float)d01;
    a.mpp = cfg->info_type == 0 ? (double)marker_size / d01 : 1.0;  // marker_meter_per_pix (:132-136)
    const bool enough = (marker_size > 0 && cfg->info_type == 0) || cfg->info_type == 1;
    a.pose = K && enough ? 1 : 0;
    const float zeros[5] = {0, 0, 0, 0, 0};
    a.cam = make_camera(K, D ? D : zeros);
    a.n_cfg = cfg->n_markers;
    a.repj_err_thres = repj_err_thres;
    a.set_y_perp = set_y_perp;
    return a;
}

static bool board_config_ok(const ab_board_config* cfg) {
    return cfg->n_markers > 0 && cfg->n_markers <= AB_BOARD_MAX_MARKERS && cfg->ids && cfg->corners;
}

int ab_set_board(ab_context* ctx, const ab_board_config* cfg, const float* K, const float* D, float marker_size, float repj_err_thres,
                 int set_y_perpendicular) {
    if (!ctx) return AB_E_INVALID;
    if (ctx->n_pending)  // a batch in flight reads the configuration
        return set_err(ctx, AB_E_STATE, "ab_set_board: %d batch(es) in flight, fetch them first", ctx->n_pending);
    if (cfg && !board_config_ok(cfg))
        return set_err(ctx, AB_E_INVALID, "ab_set_board: need 1..%d markers with ids and corners", AB_BOARD_MAX_MARKERS);
    cudaSetDevice(ctx->device);
    auto F = [](auto*& p) {
        if (p) cudaFree(p);
        p = nullptr;
    };
    ctx->have_board = false;
    memset(&ctx->board, 0, sizeof(ctx->board));
    F(ctx->d_board_ids);
    F(ctx->d_board_corners);
    if (!cfg) return AB_OK;
    const size_t n = (size_t)cfg->n_markers;
    CK(cudaMalloc(&ctx->d_board_ids, n * sizeof(int32_t)));
    CK(cudaMalloc(&ctx->d_board_corners, n * 12 * sizeof(float)));
    CK(cudaMemcpyAsync(ctx->d_board_ids, cfg->ids, n * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_board_corners, cfg->corners, n * 12 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));  // the caller's arrays may be freed on return
    ctx->board = board_args(cfg, K, D, marker_size, repj_err_thres, set_y_perpendicular);
    ctx->board.ids = ctx->d_board_ids;
    ctx->board.corners = ctx->d_board_corners;
    ctx->have_board = true;
    return AB_OK;
}

int ab_get_boards(ab_context* ctx, int n_frames, ab_board* boards, ab_marker* board_markers, int cap_per_frame) {
    if (!ctx || n_frames < 0 || (n_frames > 0 && !boards) || cap_per_frame < 0) return set_err(ctx, AB_E_INVALID, "ab_get_boards: bad arguments");
    if (!ctx->res_board) return set_err(ctx, AB_E_STATE, "ab_get_boards: the last batch returned ran without a board armed");
    if (n_frames != (int)ctx->res_boards.size())
        return set_err(ctx, AB_E_STATE, "ab_get_boards: the last batch returned has %d frames, not %d", (int)ctx->res_boards.size(), n_frames);
    if (board_markers) {
        if (!ctx->res_board_markers)
            return set_err(ctx, AB_E_STATE, "ab_get_boards: the markers of the last batch were not fetched (out == NULL)");
        for (int f = 0; f < n_frames; f++)
            if (ctx->res_boards[f].n_markers > cap_per_frame)
                return set_err(ctx, AB_E_CAPACITY, "frame %d matched %d board markers but cap_per_frame is %d", f, ctx->res_boards[f].n_markers,
                               cap_per_frame);
        for (int f = 0; f < n_frames; f++)
            memcpy(board_markers + (size_t)f * cap_per_frame, ctx->res_markers.data() + ctx->res_off[f],
                   sizeof(ab_marker) * (size_t)(ctx->res_off[f + 1] - ctx->res_off[f]));
    }
    if (n_frames > 0) memcpy(boards, ctx->res_boards.data(), sizeof(ab_board) * (size_t)n_frames);
    return AB_OK;
}

// the markers of one frame as a one-frame batch through k_board_batch
int ab_detect_board(ab_context* ctx, const ab_marker* markers, int n, const ab_board_config* cfg, const float* K, const float* D,
                    float marker_size, float repj_err_thres, int set_y_perp, ab_marker* board_markers, ab_board* out) {
    if (!ctx || !cfg || !out || n < 0 || (n > 0 && !markers)) return set_err(ctx, AB_E_INVALID, "ab_detect_board: bad arguments");
    // CV_Assert(BConf.objPoints.size() != 0 ...) (boarddetector.cpp:93)
    if (cfg->n_markers <= 0 || !cfg->ids || !cfg->corners) return set_err(ctx, AB_E_INVALID, "invalid BoardConfig that is empty");
    cudaSetDevice(ctx->device);
    memset(out, 0, sizeof(*out));
    BoardArgs a = board_args(cfg, K, D, marker_size, repj_err_thres, set_y_perp);
    const int cap = std::max(n, 1);
    const size_t ncfg = (size_t)cfg->n_markers;
    // one grow-only scratch block: markers | count | ids | corners | board | slots | points
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t off_n = al(sizeof(ab_marker) * cap), off_ids = off_n + al(sizeof(unsigned)), off_cor = off_ids + al(sizeof(int32_t) * ncfg),
                 off_board = off_cor + al(sizeof(float) * 12 * ncfg), off_slots = off_board + al(sizeof(ab_board)),
                 off_pts = off_slots + al(sizeof(int32_t) * cap), total = off_pts + sizeof(float) * BOARD_PTS_PER_MARKER * cap;
    if (int rc = ensure_scratch(ctx, total)) return rc;
    uint8_t* base = (uint8_t*)ctx->d_scratch;
    Batch b;
    memset(&b, 0, sizeof(b));
    b.B = 1;
    b.cap_c = cap;
    b.markers = (ab_marker*)base;
    b.n_markers = (unsigned*)(base + off_n);
    b.boards = (ab_board*)(base + off_board);
    b.board_slots = (int32_t*)(base + off_slots);
    b.board_pts = (float*)(base + off_pts);
    a.ids = (const int32_t*)(base + off_ids);
    a.corners = (const float*)(base + off_cor);
    const unsigned count = (unsigned)n;
    if (n > 0) CK(cudaMemcpyAsync(b.markers, markers, sizeof(ab_marker) * n, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(b.n_markers, &count, sizeof(count), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(base + off_ids, cfg->ids, sizeof(int32_t) * ncfg, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(base + off_cor, cfg->corners, sizeof(float) * 12 * ncfg, cudaMemcpyHostToDevice, ctx->stream));
    k_board_batch<<<1, 32, 0, ctx->stream>>>(b, a);
    CK(cudaGetLastError());
    std::vector<int32_t> slots(board_markers ? (size_t)n : 0);
    CK(cudaMemcpyAsync(ctx->h_scratch, b.boards, sizeof(ab_board), cudaMemcpyDeviceToHost, ctx->stream));
    if (!slots.empty()) CK(cudaMemcpyAsync(slots.data(), b.board_slots, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    memcpy(out, ctx->h_scratch, sizeof(*out));
    for (int i = 0; board_markers && i < out->n_markers; i++) {
        board_markers[i] = markers[slots[i]];
        board_markers[i].ssize = out->ssize;
    }
    return AB_OK;
}

// cv::calibrateCamera for n_cams cameras: the inputs are packed into one host block (one copy in), k_calibrate runs one CTA
// per camera, and the results and poses come back in one copy.
int ab_calibrate_cameras(ab_context* ctx, int n_cams, const ab_calib_camera* cams, ab_calib_result* out, double* rvecs, double* tvecs) {
    if (!ctx) return AB_E_INVALID;
    if (n_cams < 0 || n_cams > AB_CALIB_MAX_CAMERAS || (n_cams > 0 && (!cams || !out)))
        return set_err(ctx, AB_E_INVALID, "ab_calibrate_cameras: bad arguments (need 0 <= n_cams <= %d, cams and out)", AB_CALIB_MAX_CAMERAS);
    long long views = 0, points = 0;
    for (int c = 0; c < n_cams; c++) {
        const ab_calib_camera& k = cams[c];
        if (k.n_views < 0 || k.n_views > AB_CALIB_MAX_VIEWS || k.width < 0 || k.height < 0 || (k.n_views > 0 && !k.n_points))
            return set_err(ctx, AB_E_INVALID, "ab_calibrate_cameras: camera %d: bad size or view count (at most %d views)", c, AB_CALIB_MAX_VIEWS);
        long long np = 0;
        for (int v = 0; v < k.n_views; v++) {
            if (k.n_points[v] < 0 || k.n_points[v] > AB_CALIB_MAX_VIEW_POINTS)
                return set_err(ctx, AB_E_INVALID, "ab_calibrate_cameras: camera %d view %d: %d points (0..%d)", c, v, k.n_points[v],
                               AB_CALIB_MAX_VIEW_POINTS);
            np += k.n_points[v];
        }
        if (np > 0 && (!k.obj || !k.img)) return set_err(ctx, AB_E_INVALID, "ab_calibrate_cameras: camera %d: NULL points", c);
        views += k.n_views;
        points += np;
    }
    if (points > (1ll << 30)) return set_err(ctx, AB_E_INVALID, "ab_calibrate_cameras: %lld points in one call (at most 2^30)", points);
    if (ctx->n_pending) return set_err(ctx, AB_E_STATE, "ab_calibrate_cameras: %d batch(es) in flight, fetch them first", ctx->n_pending);
    if (n_cams == 0) return AB_OK;
    cudaSetDevice(ctx->device);
    // device block: cams | n_points | offset | obj | img | results | poses | workspace
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t off_np = al(sizeof(CalibCamRec) * n_cams), off_of = off_np + al(sizeof(int32_t) * views),
                 off_obj = off_of + al(sizeof(int32_t) * views), off_img = off_obj + al(sizeof(float) * 3 * points),
                 in_bytes = off_img + al(sizeof(float) * 2 * points), off_res = in_bytes,
                 off_pose = off_res + al(sizeof(ab_calib_result) * n_cams), off_ws = off_pose + al(sizeof(double) * 6 * views),
                 total = off_ws + sizeof(CalibView) * views;
    std::vector<uint8_t> h(off_ws);
    CalibCamRec* rec = (CalibCamRec*)h.data();
    int32_t *np = (int32_t*)(h.data() + off_np), *of = (int32_t*)(h.data() + off_of);
    float *obj = (float*)(h.data() + off_obj), *img = (float*)(h.data() + off_img);
    int v0 = 0, p0 = 0;
    for (int c = 0; c < n_cams; c++) {
        const ab_calib_camera& k = cams[c];
        rec[c] = CalibCamRec{k.width, k.height, k.n_views, v0};
        int n = 0;
        for (int v = 0; v < k.n_views; v++) {
            np[v0 + v] = k.n_points[v];
            of[v0 + v] = p0 + n;
            n += k.n_points[v];
        }
        if (n > 0) {
            memcpy(obj + 3 * (size_t)p0, k.obj, sizeof(float) * 3 * n);
            memcpy(img + 2 * (size_t)p0, k.img, sizeof(float) * 2 * n);
        }
        v0 += k.n_views;
        p0 += n;
    }
    if (int rc = ensure_scratch(ctx, total)) return rc;
    uint8_t* base = (uint8_t*)ctx->d_scratch;
    CK(cudaMemcpyAsync(base, h.data(), in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    CalibArgs a;
    a.cams = (const CalibCamRec*)base;
    a.n_points = (const int32_t*)(base + off_np);
    a.offset = (const int32_t*)(base + off_of);
    a.obj = (const float*)(base + off_obj);
    a.img = (const float*)(base + off_img);
    a.out = (ab_calib_result*)(base + off_res);
    a.poses = (double*)(base + off_pose);
    a.ws = (CalibView*)(base + off_ws);
    k_calibrate<<<n_cams, CALIB_THREADS, 0, ctx->stream>>>(a);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h.data(), base + off_res, off_ws - off_res, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    memcpy(out, h.data(), sizeof(ab_calib_result) * n_cams);
    const double* poses = (const double*)(h.data() + (off_pose - off_res));
    for (long long v = 0; v < views; v++)
        for (int i = 0; i < 3; i++) {
            if (rvecs) rvecs[3 * v + i] = poses[6 * v + i];
            if (tvecs) tvecs[3 * v + i] = poses[6 * v + 3 + i];
        }
    return AB_OK;
}

// cv::stereoCalibrate (CALIB_FIX_INTRINSIC) for n_pairs camera pairs, laid out as ab_calibrate_cameras: one host block in, one
// CTA per pair (k_stereo_calibrate), results, poses and per-view errors back in one copy.
int ab_stereo_calibrate(ab_context* ctx, int n_pairs, const ab_stereo_pair* pairs, int max_iter, double eps, ab_stereo_result* out,
                        double* rvecs, double* tvecs, double* per_view_errors) {
    if (!ctx) return AB_E_INVALID;
    if (n_pairs < 0 || n_pairs > AB_CALIB_MAX_CAMERAS || (n_pairs > 0 && (!pairs || !out)))
        return set_err(ctx, AB_E_INVALID, "ab_stereo_calibrate: bad arguments (need 0 <= n_pairs <= %d, pairs and out)", AB_CALIB_MAX_CAMERAS);
    if (max_iter < 1 || max_iter > 1000 || !(eps >= 0) || !(eps - eps == 0))
        return set_err(ctx, AB_E_INVALID, "ab_stereo_calibrate: bad criteria (need 1 <= max_iter <= 1000 and finite eps >= 0)");
    long long views = 0, points = 0;
    for (int c = 0; c < n_pairs; c++) {
        const ab_stereo_pair& k = pairs[c];
        if (k.n_views < 0 || k.n_views > AB_CALIB_MAX_VIEWS || (k.n_views > 0 && !k.n_points))
            return set_err(ctx, AB_E_INVALID, "ab_stereo_calibrate: pair %d: bad view count (at most %d views)", c, AB_CALIB_MAX_VIEWS);
        for (const double* K : {k.K1, k.K2}) {
            bool ok = K[0] > 0 && K[4] > 0;
            for (int i = 0; i < 9; i++) ok = ok && K[i] - K[i] == 0;
            if (!ok) return set_err(ctx, AB_E_INVALID, "ab_stereo_calibrate: pair %d: camera matrix not finite or fx, fy <= 0", c);
        }
        long long np = 0;
        for (int v = 0; v < k.n_views; v++) {
            if (k.n_points[v] < 0 || k.n_points[v] > AB_CALIB_MAX_VIEW_POINTS)
                return set_err(ctx, AB_E_INVALID, "ab_stereo_calibrate: pair %d view %d: %d points (0..%d)", c, v, k.n_points[v],
                               AB_CALIB_MAX_VIEW_POINTS);
            np += k.n_points[v];
        }
        if (np > 0 && (!k.obj || !k.img1 || !k.img2)) return set_err(ctx, AB_E_INVALID, "ab_stereo_calibrate: pair %d: NULL points", c);
        views += k.n_views;
        points += np;
    }
    if (points > (1ll << 30)) return set_err(ctx, AB_E_INVALID, "ab_stereo_calibrate: %lld points in one call (at most 2^30)", points);
    if (ctx->n_pending) return set_err(ctx, AB_E_STATE, "ab_stereo_calibrate: %d batch(es) in flight, fetch them first", ctx->n_pending);
    if (n_pairs == 0) return AB_OK;
    cudaSetDevice(ctx->device);
    // device block: pairs | n_points | offset | obj | img1 | img2 | results | poses | errors | workspace
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t off_np = al(sizeof(StereoPairRec) * n_pairs), off_of = off_np + al(sizeof(int32_t) * views),
                 off_obj = off_of + al(sizeof(int32_t) * views), off_i1 = off_obj + al(sizeof(float) * 3 * points),
                 off_i2 = off_i1 + al(sizeof(float) * 2 * points), in_bytes = off_i2 + al(sizeof(float) * 2 * points),
                 off_res = in_bytes, off_pose = off_res + al(sizeof(ab_stereo_result) * n_pairs),
                 off_err = off_pose + al(sizeof(double) * 6 * views), off_ws = off_err + al(sizeof(double) * 2 * views),
                 total = off_ws + sizeof(StereoView) * views;
    std::vector<uint8_t> h(off_ws);
    StereoPairRec* rec = (StereoPairRec*)h.data();
    int32_t *np = (int32_t*)(h.data() + off_np), *of = (int32_t*)(h.data() + off_of);
    float *obj = (float*)(h.data() + off_obj), *i1 = (float*)(h.data() + off_i1), *i2 = (float*)(h.data() + off_i2);
    int v0 = 0, p0 = 0;
    for (int c = 0; c < n_pairs; c++) {
        const ab_stereo_pair& k = pairs[c];
        StereoPairRec& r = rec[c];
        r.n_views = k.n_views;
        r.view0 = v0;
        memcpy(r.K1, k.K1, sizeof(r.K1));
        memcpy(r.K2, k.K2, sizeof(r.K2));
        stereo_intrinsics(k.K1, k.D1, r.kk1);
        stereo_intrinsics(k.K2, k.D2, r.kk2);
        int n = 0;
        for (int v = 0; v < k.n_views; v++) {
            np[v0 + v] = k.n_points[v];
            of[v0 + v] = p0 + n;
            n += k.n_points[v];
        }
        if (n > 0) {
            memcpy(obj + 3 * (size_t)p0, k.obj, sizeof(float) * 3 * n);
            memcpy(i1 + 2 * (size_t)p0, k.img1, sizeof(float) * 2 * n);
            memcpy(i2 + 2 * (size_t)p0, k.img2, sizeof(float) * 2 * n);
        }
        v0 += k.n_views;
        p0 += n;
    }
    if (int rc = ensure_scratch(ctx, total)) return rc;
    uint8_t* base = (uint8_t*)ctx->d_scratch;
    CK(cudaMemcpyAsync(base, h.data(), in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    StereoArgs a;
    a.pairs = (const StereoPairRec*)base;
    a.n_points = (const int32_t*)(base + off_np);
    a.offset = (const int32_t*)(base + off_of);
    a.obj = (const float*)(base + off_obj);
    a.img1 = (const float*)(base + off_i1);
    a.img2 = (const float*)(base + off_i2);
    a.max_iter = max_iter;
    a.eps = eps;
    a.out = (ab_stereo_result*)(base + off_res);
    a.poses = (double*)(base + off_pose);
    a.errs = (double*)(base + off_err);
    a.ws = (StereoView*)(base + off_ws);
    k_stereo_calibrate<<<n_pairs, CALIB_THREADS, 0, ctx->stream>>>(a);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h.data(), base + off_res, off_ws - off_res, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    memcpy(out, h.data(), sizeof(ab_stereo_result) * n_pairs);
    const double* poses = (const double*)(h.data() + (off_pose - off_res));
    const double* errs = (const double*)(h.data() + (off_err - off_res));
    for (long long v = 0; v < views; v++) {
        for (int i = 0; i < 3; i++) {
            if (rvecs) rvecs[3 * v + i] = poses[6 * v + i];
            if (tvecs) tvecs[3 * v + i] = poses[6 * v + 3 + i];
        }
        if (per_view_errors)
            for (int k = 0; k < 2; k++) per_view_errors[2 * v + k] = errs[2 * v + k];
    }
    return AB_OK;
}

int ab_host_alloc(void** ptr, size_t bytes) {
    if (!ptr) return AB_E_INVALID;
    return cudaMallocHost(ptr, bytes) == cudaSuccess ? AB_OK : AB_E_CUDA;
}

int ab_host_free(void* ptr) { return cudaFreeHost(ptr) == cudaSuccess ? AB_OK : AB_E_CUDA; }

}  // extern "C"
