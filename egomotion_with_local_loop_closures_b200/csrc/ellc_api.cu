// ellc_api.cu -- C-ABI implementation (include/ellc_gn.h): handle, device pools, batching and launch orchestration.
//
// Device memory layout (all pools are slot-major, one cudaMalloc each):
//   frames     img : u8   pyramid levels 0..3 concatenated (cv::pyrDown dims)          slot stride = geo.img_off[4]
//              tex : u32  packed texels, level windows concatenated                    slot stride = geo.win_off[4]
//   keyframes  img : u8   as frames
//              depth, var : f32 level windows concatenated                             slot stride = geo.win_off[4]
//              mask : u8  level windows                                                  "
//              sel_geo : SelGeo[ ] + sel_pix : SelPix[ ] compacted selected pixels, level l at win_off[l]
//              count[4], rowcount / rowoff scratch
// Uploads only mark slots dirty; the pyramid / texel / selection kernels run batched over all dirty slots right before
// the next consumer (track, evaluate, read-back) -- a whole batch costs 4 (frames) + 6 (keyframes) launches.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "ellc_internal.h"
#include "ellc_lie.cuh"

using namespace ellc;

// ---- multi-GPU result exchange (SURVEY 8e; include/ellc_gn.h "result exchange") ------------------------------------------------
// Every rank owns one block of device memory: a header of counters and a ring of kXchgRing result tables of `capacity` records.
// Token t (the t-th exchanged batch, the same number on every rank) uses table t % kXchgRing everywhere.  A sender's tracking
// kernel stores its records into the tables of the receiving ranks (peer memory mapped with CUDA IPC or, inside one process,
// cudaDeviceEnablePeerAccess) and a one-warp kernel behind it adds its record count to the receivers' arrived[] counters; a
// receiver's HOST polls its own counter, copies the table out and publishes released[0] = t, which a sender reads (from the
// receiver's memory) before it reuses that table for token t + kXchgRing.  No kernel ever spins.
// The release is published by a one-thread kernel on the receiver's TRACKING stream, in front of its next batch (or at once
// when no batch is queued).  Measured at N = 2: the same kernel on the download stream has to find a free CTA slot among the
// pending CTAs of the highest-priority tracking kernel (the receiving rank lost 0.5-0.8 ms per step and its e2e uploads could
// not overlap the running batch); an 8-byte cudaMemcpyAsync into the block instead waits for the whole running kernel (25 ms
// per step instead of 14).  At a batch boundary the GPU is free and the release costs nothing.
constexpr int kXchgRing = 4;
struct XchgHeader {
    unsigned long long arrived[kXchgRing];             // records delivered into table r, cumulative over the tokens that used it
    unsigned long long released[kXchgRing];            // [0]: last token whose table the owner has finished copying out (tokens are
                                                       // consumed in order); [1..]: unused
    unsigned long long pad[32 - 2 * kXchgRing];
};
static_assert(sizeof(XchgHeader) == 256, "exchange header is one 256-byte record");
struct ellc_exchange {
    int rank, world, capacity;
    void* block;                                       // own block (cudaMalloc)
    void* peer_block[ELLC_MAX_RANKS];                  // every rank's block as mapped into this process (own: block)
    bool peer_ipc[ELLC_MAX_RANKS];                     // opened with cudaIpcOpenMemHandle
    bool attached;
    long long token;                                   // tokens issued so far
    unsigned long long expected[kXchgRing];            // records expected in the own table r, cumulative
    struct Tok { long long seq; int n, n_total, root; } tok[kXchgRing];
    unsigned long long** d_ctr;                        // device array [kXchgRing][ELLC_MAX_RANKS]: &header(d)->arrived[r]
    unsigned long long* h_poll;                        // pinned scratch of the host polls
    long long consumed, published;                     // last token copied out by this rank / last one written to released[0]
};
struct ellc_handle {
    ellc_config cfg;
    Geometry geo;
    LevelK K[kLevels];
    int rows_total;
    cudaStream_t stream;                               // main compute stream: prepare kernels, evaluate, read-backs, small staging copies
    cudaStream_t tstream[2];                           // tracking kernels: batch `seq` runs on tstream[seq & 1], ordered behind batch seq - 1
                                                       // by its completion event (or not, ELLC_OVERLAP=1: measured slower, see ellc_create);
                                                       // both at the highest priority.  Keeping the batches off the main stream lets
                                                       // synchronous main-stream calls (evaluate, read-backs) be ordered explicitly
    cudaEvent_t main_ev;                               // recorded on the main stream at every batch launch; the batch's stream waits for it
    cudaEvent_t hyp_ev; bool hyp_pending;              // depth pyramids built from hypotheses on the main stream (prep stream must wait)
    bool overlap_batches;                              // consecutive forward batches overlap at their tails (default; ELLC_OVERLAP=0 serialises them: A/B measurement)
    cudaStream_t copy_stream;                          // H2D uploads of images / depth / variance (overlap with compute)
    cudaStream_t d2h_stream;                           // result downloads of finished batches
    cudaEvent_t ev0r[4], ev1r[4];                      // track-kernel timing events of the last four batches (index: sequence & 3)
    cudaEvent_t up_ev;                                 // re-recorded after every upload on copy_stream
    cudaStream_t prep_stream;                          // preparation of freshly uploaded slots (overlaps the previous batch's kernels)
    cudaEvent_t prep_ev;                               // recorded after every such preparation; the compute stream waits for it
    int* d_slots_p;                                    // slot lists of the preparation stream (2 x slots_cap)
    bool uploads_pending;
    cudaEvent_t batch_ev[4];                           // completion of the last 4 track batches (ring by sequence number)
    long long batch_seq, batch_done_seq;               // last enqueued / last known-complete batch
    std::vector<long long> fr_reader, kf_reader;       // sequence number of the last batch that reads each slot
    bool ev_valid;
    // pools
    uint8_t* fr_img; uint32_t* fr_tex;
    uint8_t* kf_img; float* kf_depth; float* kf_var; uint8_t* kf_mask; SelGeo* kf_geo; SelPix* kf_pix; float* kf_ikf;
    float* fr_hist;                                    // [frame slot][256] normalised histograms (loop-closure gating), lazy
    std::vector<char> fr_hist_ready;
    // hypothesis staging of ellc_upload_keyframe_hypotheses (allocated on first use) and per-slot valid counts
    uint8_t* d_hyp; int* d_nvalid;
    std::vector<int> kf_nvalid;                        // -1: not uploaded from hypotheses / not fetched yet
    // loop-closure state, allocated on first use (ensure_lc_pools)
    float* fr_weight; float* kf_weight; LcRec* kf_lc; float* kf_lcH; float4* kf_lcf; uint32_t* kf_lcp;
    std::vector<int> kf_wcount;                        // numWeightsAdded[level] per keyframe slot
    std::vector<char> kf_lc_ready;                     // LcRec / hessian built for the slot's current contents
    int* kf_count; int* kf_rowcount; int* kf_rowoff;
    std::vector<uint8_t> fr_state, kf_state;          // 0 empty, 1 image present (dirty), 2 prepared
    std::vector<int> fr_dirty, kf_dirty;
    // staging
    int* d_slots; int slots_cap;
    // per-batch staging / result buffers: ring of 4 by sequence number (two batches may be in flight, a third being staged, and the
    // records of a finished one still being downloaded); entry r is reused by batch seq+4 after batch seq has completed
    ellc_pair* d_pairs4[4]; ellc_result* d_results4[4]; int* d_order4[4]; int* d_gidx4[4]; int ring_cap[4]; long long res_seq[4];
    bool res_taken[4];                                 // the records of the entry's last batch have been copied out (the entry may be regrown)
    ellc_pair* d_pairs; ellc_result* d_results; int* d_order;       // entry of the batch being launched / launched last
    ellc_result* d_eval_result;                        // ellc_gn_evaluate's own record (never clobbers an undownloaded batch)
    ellc_exchange* xc;                                 // multi-GPU result exchange (ellc_exchange_create), or null
    // device-side loop-closure pair list (ellc_lc_generate_pairs): one allocation carved into ring / queries / per-query segments /
    // packed list / statistics / query index / total
    char* d_gen; size_t gen_bytes; int gen_cap_q, gen_cap_ring;
    ellc_pair* d_gen_pairs; int gen_n, gen_flags;
    std::vector<int> gen_kf_slots, gen_frame_slots;    // slots the generated pairs may read (slot-reuse bookkeeping)
    ellc_iter_trace* d_trace; int64_t trace_cap;
    char* d_seq; size_t seq_bytes;                     // buffer of ellc_track_sequence_steps (steps, order, pairs, records, world poses)
    float* d_small;                                    // 128 floats in/out for solve_update
    float* d_weight; int64_t weight_cap;
    void* h_pin; void* d_pin; size_t pin_cap, pin_used;             // pinned bump arena for small H2D payloads
    // camera ingestion (ellc_set_camera): resize taps, undistortion map at the tap positions, per-call job list, staging of host
    // camera images; ingest_ev orders the copy stream -> ingest kernel (preparation stream) -> copy stream chain
    bool cam_set; IngestGeo cam_geo;
    int4* d_cam_cols; int4* d_cam_rows; uint2* d_cam_map; IngestJob* d_ingest_jobs;
    uint8_t* d_cam_stage; size_t cam_stage_cap;
    cudaEvent_t ingest_ev;
    std::string err;
    int64_t launches;
};

static thread_local std::string g_create_err;

#define CU_TRY(h, call)                                                                              \
    do {                                                                                             \
        cudaError_t e__ = (call);                                                                    \
        if (e__ != cudaSuccess) {                                                                    \
            (h)->err = std::string(#call) + ": " + cudaGetErrorString(e__);                          \
            return ELLC_ERR_CUDA;                                                                    \
        }                                                                                            \
    } while (0)

static void build_geometry(const ellc_config& c, Geometry& g) {
    g.width = c.width; g.height = c.height;
    int pw = c.width, ph = c.height;
    g.img_off[0] = 0; g.win_off[0] = 0;
    for (int l = 0; l < kLevels; ++l) {
        g.pyr_w[l] = pw; g.pyr_h[l] = ph;
        g.cols[l] = c.width >> l; g.rows[l] = c.height >> l;
        g.img_off[l + 1] = g.img_off[l] + (int64_t)pw * ph;
        g.win_off[l + 1] = g.win_off[l] + (int64_t)g.cols[l] * g.rows[l];
        pw = (pw + 1) / 2; ph = (ph + 1) / 2;
    }
}

// GetIntrinsic, src/UserDefinedFunc.cpp:33-49
static void build_intrinsics(const ellc_config& c, LevelK K[kLevels]) {
    for (int l = 0; l < kLevels; ++l) {
        const double s = (double)(1 << l);
        K[l].fx = (float)(c.fx / s); K[l].fy = (float)(c.fy / s);
        K[l].cx = (float)(c.cx / s) + 0.0f; K[l].cy = (float)(c.cy / s) + 0.0f;   // + 0.0f: never -0.0 (bit-pattern bound tests)
        K[l].ifx = 1.0f / K[l].fx; K[l].ify = 1.0f / K[l].fy;
        K[l].fy_ifx = K[l].fy / K[l].fx; K[l].fx_ify = K[l].fx / K[l].fy;
        K[l].cm1 = (float)((c.width >> l) - 1); K[l].rm1 = (float)((c.height >> l) - 1);
        const float bounds[4] = {(float)(c.width >> l), K[l].cm1, (float)(c.height >> l), K[l].rm1};
        uint32_t bits[4];
        std::memcpy(bits, bounds, sizeof(bits));
        K[l].colsf_bits = bits[0]; K[l].cm1_bits = bits[1]; K[l].rowsf_bits = bits[2]; K[l].rm1_bits = bits[3];
    }
}

static void exchange_release(ellc_handle* h);

extern "C" {

#ifndef ELLC_SRC_HASH
#define ELLC_SRC_HASH "unknown"
#endif
const char* ellc_version(void) { return "ellc-gn-b200 0.2 (sm_100a) src:" ELLC_SRC_HASH; }

void ellc_default_config(ellc_config* c, int32_t width, int32_t height) {
    std::memset(c, 0, sizeof(*c));
    c->width = width; c->height = height;
    c->fx = 0.8f * width; c->fy = 0.8f * width; c->cx = width / 2.0f; c->cy = height / 2.0f;
    c->max_iter[0] = 4; c->max_iter[1] = 7; c->max_iter[2] = 9; c->max_iter[3] = 12;      // src/main.cpp:34
    c->huber_d = 3.0f; c->camera_pixel_noise_2 = 4.0f * 4.0f;                             // src/ExternVariable.h:148-149
    c->weight[0] = c->weight[1] = c->weight[2] = 100000.0f;                               // :76
    c->weight[3] = c->weight[4] = c->weight[5] = 10000.0f;
    c->stop_threshold = 1.0f;                                                             // src/ImageFunc.cpp:251
    c->arithmetic = ELLC_ARITH_FAST;
    c->jacobian_at_warped = 0;
    c->max_keyframes = 8; c->max_frames = 64;
    c->ctas_per_pair = 0; c->device = 0;
    c->lm_lambda = 0.0f; c->lm_up = 4.0f; c->lm_down = 0.5f;                              // 0 = the reference's plain Gauss-Newton step
    c->lc_bands = 2;                                                                      // FLAG_DO_PARALLEL_CONST_WEIGHT_POSE_EST
}

const char* ellc_last_error_string(const ellc_handle* h) { return h ? h->err.c_str() : g_create_err.c_str(); }

int ellc_destroy(ellc_handle* h) {
    if (!h) return ELLC_OK;
    cudaSetDevice(h->cfg.device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    for (int i = 0; i < 2; ++i) if (h->tstream[i]) cudaStreamSynchronize(h->tstream[i]);
    if (h->prep_stream) cudaStreamSynchronize(h->prep_stream);
    exchange_release(h);
    if (h->copy_stream) cudaStreamSynchronize(h->copy_stream);
    if (h->d2h_stream) cudaStreamSynchronize(h->d2h_stream);
    cudaFree(h->fr_img); cudaFree(h->fr_tex); cudaFree(h->kf_img); cudaFree(h->kf_depth); cudaFree(h->kf_var);
    cudaFree(h->kf_mask); cudaFree(h->kf_geo); cudaFree(h->kf_pix); cudaFree(h->kf_ikf);
    cudaFree(h->d_hyp); cudaFree(h->d_nvalid); cudaFree(h->fr_hist);
    cudaFree(h->fr_weight); cudaFree(h->kf_weight); cudaFree(h->kf_lc); cudaFree(h->kf_lcH); cudaFree(h->kf_lcf); cudaFree(h->kf_lcp); cudaFree(h->kf_count); cudaFree(h->kf_rowcount); cudaFree(h->kf_rowoff);
    cudaFree(h->d_slots); cudaFree(h->d_slots_p); cudaFree(h->d_trace); cudaFree(h->d_small); cudaFree(h->d_eval_result); cudaFree(h->d_gen);
    cudaFree(h->d_seq);
    for (int r = 0; r < 4; ++r) { cudaFree(h->d_pairs4[r]); cudaFree(h->d_results4[r]); cudaFree(h->d_order4[r]); cudaFree(h->d_gidx4[r]); }
    cudaFree(h->d_weight);
    cudaFree(h->d_cam_cols); cudaFree(h->d_cam_rows); cudaFree(h->d_cam_map); cudaFree(h->d_ingest_jobs); cudaFree(h->d_cam_stage);
    if (h->h_pin) cudaFreeHost(h->h_pin);
    if (h->ev_valid) {
        for (int i = 0; i < 4; ++i) { cudaEventDestroy(h->ev0r[i]); cudaEventDestroy(h->ev1r[i]); }
        cudaEventDestroy(h->up_ev); cudaEventDestroy(h->prep_ev); cudaEventDestroy(h->main_ev); cudaEventDestroy(h->hyp_ev);
        cudaEventDestroy(h->ingest_ev);
        for (int i = 0; i < 4; ++i) cudaEventDestroy(h->batch_ev[i]);
    }
    if (h->stream) cudaStreamDestroy(h->stream);
    for (int i = 0; i < 2; ++i) if (h->tstream[i]) cudaStreamDestroy(h->tstream[i]);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->d2h_stream) cudaStreamDestroy(h->d2h_stream);
    if (h->prep_stream) cudaStreamDestroy(h->prep_stream);
    delete h;
    return ELLC_OK;
}

int ellc_create(const ellc_config* cfg, ellc_handle** out) {
    if (!cfg || !out) { g_create_err = "null argument"; return ELLC_ERR_INVALID; }
    *out = nullptr;
    if (cfg->width < 16 || cfg->height < 16 || cfg->width > 2047 || cfg->height > 2047 || cfg->max_keyframes < 1 ||
        cfg->max_frames < 1) { g_create_err = "unsupported size / slot count"; return ELLC_ERR_INVALID; }
    if (cfg->jacobian_at_warped && cfg->arithmetic != ELLC_ARITH_STRICT) {
        g_create_err = "jacobian_at_warped (Pyramid.cpp variant) is built in the ELLC_ARITH_STRICT flavour only"; return ELLC_ERR_INVALID;
    }
    for (int l = 0; l < kLevels; ++l)
        if (cfg->max_iter[l] < 0) { g_create_err = "negative max_iter"; return ELLC_ERR_INVALID; }
    if (cfg->arithmetic < ELLC_ARITH_FAST || cfg->arithmetic > ELLC_ARITH_REFERENCE) { g_create_err = "unknown arithmetic flavour"; return ELLC_ERR_INVALID; }
    if (cfg->arithmetic == ELLC_ARITH_REFERENCE) {
        // the reference's summation order is built for one CTA per pair, the PixelWisePyramid.cpp Jacobian and the plain step
        if (cfg->jacobian_at_warped) { g_create_err = "ELLC_ARITH_REFERENCE does not cover the Pyramid.cpp variant (jacobian_at_warped)"; return ELLC_ERR_INVALID; }
        if (cfg->lm_lambda != 0.0f) { g_create_err = "ELLC_ARITH_REFERENCE takes the reference's undamped step (lm_lambda = 0)"; return ELLC_ERR_INVALID; }
        if (cfg->ctas_per_pair != 0 && cfg->ctas_per_pair != 1) { g_create_err = "ELLC_ARITH_REFERENCE tracks a pair on one CTA (ctas_per_pair 0 or 1)"; return ELLC_ERR_INVALID; }
        if (cfg->pairs_per_cta != 0 && cfg->pairs_per_cta != 1) { g_create_err = "ELLC_ARITH_REFERENCE tracks one pair per CTA (pairs_per_cta 0 or 1)"; return ELLC_ERR_INVALID; }
        if (cfg->lc_bands != 1 && cfg->lc_bands != 2) { g_create_err = "lc_bands must be 1 or 2"; return ELLC_ERR_INVALID; }
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev <= cfg->device) {
        g_create_err = std::string("no usable CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e);
        return ELLC_ERR_CUDA;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess || prop.major < 10) {
        g_create_err = "device is not sm_100-class (this library carries sm_100a code only)";
        return ELLC_ERR_CUDA;
    }
    ellc_handle* h = new (std::nothrow) ellc_handle();
    if (!h) { g_create_err = "out of host memory"; return ELLC_ERR_INVALID; }
    h->cfg = *cfg;
    build_geometry(*cfg, h->geo);
    build_intrinsics(*cfg, h->K);
    h->rows_total = 0;
    for (int l = 0; l < kLevels; ++l) h->rows_total += h->geo.rows[l];
    h->fr_state.assign(cfg->max_frames, 0);
    h->kf_state.assign(cfg->max_keyframes, 0);
    h->launches = 0;
#define CR_TRY(call)                                                                                 \
    do {                                                                                             \
        cudaError_t e__ = (call);                                                                    \
        if (e__ != cudaSuccess) {                                                                    \
            g_create_err = std::string(#call) + ": " + cudaGetErrorString(e__);                      \
            ellc_destroy(h);                                                                         \
            return ELLC_ERR_CUDA;                                                                    \
        }                                                                                            \
    } while (0)
    CR_TRY(cudaSetDevice(cfg->device));
    // The tracking kernels get the highest CTA-scheduling priority, the preparation stream the lowest: preparation of the next
    // batch runs in the SM time the tracking kernel of the current one leaves over (mostly its last wave) instead of slowing it down.
    int prio_least = 0, prio_greatest = 0;
    CR_TRY(cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest));
    CR_TRY(cudaStreamCreateWithPriority(&h->stream, cudaStreamNonBlocking, prio_greatest));
    for (int i = 0; i < 2; ++i) CR_TRY(cudaStreamCreateWithPriority(&h->tstream[i], cudaStreamNonBlocking, prio_greatest));
    // MEASURED (round 2, 4608 pairs per batch): letting batch k+1 start while batch k still runs does NOT just fill its last wave --
    // its CTAs are dispatched as soon as its preparation is done, the two batches then share the SMs for most of their run time
    // with two different working sets in L2: 270k tracks/s against 335k with the batches serialised.  Off unless ELLC_OVERLAP=1.
    h->overlap_batches = true;
    if (const char* e = std::getenv("ELLC_OVERLAP")) h->overlap_batches = (*e == '1');
    CR_TRY(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    CR_TRY(cudaStreamCreateWithFlags(&h->d2h_stream, cudaStreamNonBlocking));
    CR_TRY(cudaStreamCreateWithPriority(&h->prep_stream, cudaStreamNonBlocking, prio_least));
    for (int i = 0; i < 4; ++i) { CR_TRY(cudaEventCreate(&h->ev0r[i])); CR_TRY(cudaEventCreate(&h->ev1r[i])); }
    CR_TRY(cudaEventCreateWithFlags(&h->up_ev, cudaEventDisableTiming));
    CR_TRY(cudaEventCreateWithFlags(&h->prep_ev, cudaEventDisableTiming));
    CR_TRY(cudaEventCreateWithFlags(&h->main_ev, cudaEventDisableTiming));
    CR_TRY(cudaEventCreateWithFlags(&h->hyp_ev, cudaEventDisableTiming));
    CR_TRY(cudaEventCreateWithFlags(&h->ingest_ev, cudaEventDisableTiming));
    for (int i = 0; i < 4; ++i) CR_TRY(cudaEventCreateWithFlags(&h->batch_ev[i], cudaEventDisableTiming));
    h->ev_valid = true;
    h->fr_reader.assign(cfg->max_frames, 0);
    h->kf_wcount.assign((size_t)cfg->max_keyframes * kLevels, 0);
    h->kf_lc_ready.assign(cfg->max_keyframes, 0);
    h->kf_nvalid.assign(cfg->max_keyframes, -1);
    h->fr_hist_ready.assign(cfg->max_frames, 0);
    h->kf_reader.assign(cfg->max_keyframes, 0);
    const int64_t img = h->geo.img_off[kLevels], win = h->geo.win_off[kLevels];
    const int64_t nf = cfg->max_frames, nk = cfg->max_keyframes;
    CR_TRY(cudaMalloc(&h->fr_img, nf * img));
    CR_TRY(cudaMalloc(&h->fr_tex, (nf * (win + kTexPad) + kTexTail) * sizeof(uint32_t)));
    CR_TRY(cudaMemsetAsync(h->fr_tex, 0, (nf * (win + kTexPad) + kTexTail) * sizeof(uint32_t), h->stream));   // pack_tex writes the pad words
    CR_TRY(cudaMalloc(&h->kf_img, nk * img));
    CR_TRY(cudaMalloc(&h->kf_depth, nk * win * sizeof(float)));
    CR_TRY(cudaMalloc(&h->kf_var, nk * win * sizeof(float)));
    CR_TRY(cudaMalloc(&h->kf_mask, nk * win));
    CR_TRY(cudaMalloc(&h->kf_geo, (nk * win + kRecTail) * sizeof(SelGeo)));
    CR_TRY(cudaMalloc(&h->kf_pix, (nk * win + kRecTail) * sizeof(SelPix)));
    CR_TRY(cudaMalloc(&h->kf_ikf, (nk * win + kRecTail) * sizeof(float)));
    CR_TRY(cudaMemsetAsync(h->kf_geo, 0, (nk * win + kRecTail) * sizeof(SelGeo), h->stream));
    CR_TRY(cudaMemsetAsync(h->kf_ikf, 0, (nk * win + kRecTail) * sizeof(float), h->stream));
    CR_TRY(cudaMalloc(&h->kf_count, nk * kLevels * sizeof(int)));
    CR_TRY(cudaMalloc(&h->kf_rowcount, nk * h->rows_total * sizeof(int)));
    CR_TRY(cudaMalloc(&h->kf_rowoff, nk * h->rows_total * sizeof(int)));
    h->slots_cap = (int)(nf > nk ? nf : nk);
    CR_TRY(cudaMalloc(&h->d_slots, 2 * h->slots_cap * sizeof(int)));
    CR_TRY(cudaMalloc(&h->d_slots_p, 2 * h->slots_cap * sizeof(int)));
    CR_TRY(cudaMalloc(&h->d_small, 128 * sizeof(float)));
    CR_TRY(cudaMalloc(&h->d_eval_result, sizeof(ellc_result) + 256));
    h->pin_cap = 32 << 20;
    CR_TRY(cudaHostAlloc(&h->h_pin, h->pin_cap, cudaHostAllocMapped));
    CR_TRY(cudaHostGetDevicePointer(&h->d_pin, h->h_pin, 0));
    h->pin_used = 0;
    CR_TRY(cudaMemsetAsync(h->kf_count, 0, nk * kLevels * sizeof(int), h->stream));
    CR_TRY(cudaStreamSynchronize(h->stream));
#undef CR_TRY
    *out = h;
    return ELLC_OK;
}

}  // extern "C"

// ---- internal helpers ------------------------------------------------------------------------------------------------
// Copy a small host payload to the device through the pinned arena (no implicit host/device serialisation).  The arena is a bump
// allocator that is only ever rewound after EVERY stream that may still pull from it has been synchronised (here, when it is
// full, and in ellc_synchronize): a pull kernel enqueued on the low-priority preparation stream, or behind an event on a tracking
// stream, can run long after the call that staged its bytes has returned.
static int sync_all_streams(ellc_handle* h) {
    CU_TRY(h, cudaStreamSynchronize(h->copy_stream));
    CU_TRY(h, cudaStreamSynchronize(h->prep_stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    for (int i = 0; i < 2; ++i) CU_TRY(h, cudaStreamSynchronize(h->tstream[i]));
    CU_TRY(h, cudaStreamSynchronize(h->d2h_stream));
    h->batch_done_seq = h->batch_seq;
    h->pin_used = 0;
    return ELLC_OK;
}
static int stage_h2d_on(ellc_handle* h, cudaStream_t st, void* dst, const void* src, size_t bytes) {
    if (bytes > h->pin_cap / 4) {           // large payload: plain (staged) async copy
        CU_TRY(h, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
        return ELLC_OK;
    }
    const size_t aligned = (bytes + 255) & ~(size_t)255;
    if (h->pin_used + aligned > h->pin_cap) {
        int rc = sync_all_streams(h);
        if (rc) return rc;
    }
    void* p = (char*)h->h_pin + h->pin_used;
    std::memcpy(p, src, bytes);
    h->pin_used += aligned;
    // pulled by the SMs, not the copy engine: see pull_host_words_kernel
    h->launches += launch_pull_host(st, dst, (char*)h->d_pin + ((char*)p - (char*)h->h_pin), bytes);
    CU_TRY(h, cudaGetLastError());
    return ELLC_OK;
}
static int stage_h2d(ellc_handle* h, void* dst, const void* src, size_t bytes) { return stage_h2d_on(h, h->stream, dst, src, bytes); }

// batch_done_seq: every batch up to and including this sequence number is known to be complete
static void note_done(ellc_handle* h, long long seq) {
    if (seq == h->batch_done_seq + 1) h->batch_done_seq = seq;
}
// Work on the main stream that reads or writes slot data is ordered behind the (up to two) tracking batches in flight on the
// tracking streams.  The pipelined preparation paths (flush_dirty's side path, ellc_prepare_async) do NOT call this: they order
// themselves behind the last batch that READ their slots only.
static int main_waits_batches(ellc_handle* h) {
    for (long long q = h->batch_seq; q >= 1 && q > h->batch_seq - 2; --q)
        if (q > h->batch_done_seq) CU_TRY(h, cudaStreamWaitEvent(h->stream, h->batch_ev[q & 3], 0));
    return ELLC_OK;
}

// An upload overwrites a slot on copy_stream.  It must not pass a track batch that still reads the slot:
// wait for that batch's completion event, unless it is already known to be finished.
static int guard_slot_write(ellc_handle* h, long long reader_seq) {
    if (reader_seq <= h->batch_done_seq) return ELLC_OK;
    if (reader_seq + 4 <= h->batch_seq) return ELLC_OK;                        // ring entry recycled => that batch was waited for
    CU_TRY(h, cudaStreamWaitEvent(h->copy_stream, h->batch_ev[reader_seq & 3], 0));
    return ELLC_OK;
}
static int after_upload(ellc_handle* h) {
    CU_TRY(h, cudaEventRecord(h->up_ev, h->copy_stream));
    h->uploads_pending = true;
    return ELLC_OK;
}

// Ring entry r = seq & 3 of the per-batch buffers; the caller has already waited for batch seq - 4, the previous user of the entry.
// Growing it frees that batch's records: a pointer returned by ellc_track_batch_async is valid until three more batches have
// been launched (include/ellc_gn.h).
static int grow_ring_entry(ellc_handle* h, int r, int cap) {
    cudaFree(h->d_pairs4[r]); cudaFree(h->d_results4[r]); cudaFree(h->d_order4[r]); cudaFree(h->d_gidx4[r]);
    h->d_pairs4[r] = nullptr; h->d_results4[r] = nullptr; h->d_order4[r] = nullptr; h->d_gidx4[r] = nullptr; h->ring_cap[r] = 0;
    CU_TRY(h, cudaMalloc(&h->d_pairs4[r], (size_t)cap * sizeof(ellc_pair)));
    CU_TRY(h, cudaMalloc(&h->d_results4[r], (size_t)cap * sizeof(ellc_result)));
    CU_TRY(h, cudaMalloc(&h->d_order4[r], (size_t)cap * sizeof(int)));
    CU_TRY(h, cudaMalloc(&h->d_gidx4[r], (size_t)cap * sizeof(int)));
    h->ring_cap[r] = cap;
    return ELLC_OK;
}
// (Re)allocation of a ring entry is a cudaFree + cudaMalloc, i.e. an implicit device synchronisation plus milliseconds of driver time.
// It must not trickle in one entry per batch (measured: the FOURTH batch of a new size, the first to reuse entry 0, stalled the
// caller's pipelined loop for 1 - 185 ms): when one entry has to grow, every other entry that is idle -- never used, or its last
// batch complete and its records copied out -- grows with it.
static int ensure_ring_cap(ellc_handle* h, int r, int n, bool want_trace) {
    if (n > h->ring_cap[r]) {
        const int cap = n < 256 ? 256 : n;
        int rc = grow_ring_entry(h, r, cap);
        if (rc) return rc;
        for (int q = 0; q < 4; ++q) {
            const bool idle = h->res_seq[q] == 0 || (h->res_seq[q] <= h->batch_done_seq && h->res_taken[q]);
            if (q != r && h->ring_cap[q] < cap && idle) { rc = grow_ring_entry(h, q, cap); if (rc) return rc; }
        }
    }
    if (want_trace) {
        const int64_t need = (int64_t)n * kLevels * ELLC_MAX_TRACE_ITERS;
        if (need > h->trace_cap) {
            cudaFree(h->d_trace); h->d_trace = nullptr; h->trace_cap = 0;
            CU_TRY(h, cudaMalloc(&h->d_trace, (size_t)need * sizeof(ellc_iter_trace)));
            h->trace_cap = need;
        }
    }
    return ELLC_OK;
}

// side = true: on the preparation stream with its own slot lists (freshly uploaded slots, see flush_dirty)
static int prepare_frames_impl(ellc_handle* h, int n, const int* slots, bool side = false) {
    if (n <= 0) return ELLC_OK;
    cudaStream_t st = side ? h->prep_stream : h->stream;
    int* d_slots = side ? h->d_slots_p : h->d_slots;
    int rc = side ? ELLC_OK : main_waits_batches(h);
    if (rc) return rc;
    rc = stage_h2d_on(h, st, d_slots, slots, (size_t)n * sizeof(int));
    if (rc) return rc;
    h->launches += launch_pyramid(st, h->fr_img, h->geo.img_off[kLevels], d_slots, n, h->geo);
    h->launches += launch_pack_tex(st, h->fr_img, h->geo.img_off[kLevels], h->fr_tex, h->geo.win_off[kLevels] + kTexPad,
                                   d_slots, n, h->geo);
    CU_TRY(h, cudaGetLastError());
    for (int i = 0; i < n; ++i) h->fr_state[slots[i]] = 2;
    return ELLC_OK;
}

static int prepare_keyframes_impl(ellc_handle* h, int n, const int* slots, bool side = false) {
    if (n <= 0) return ELLC_OK;
    cudaStream_t st = side ? h->prep_stream : h->stream;
    int* d_slots = (side ? h->d_slots_p : h->d_slots) + h->slots_cap;
    int rc = side ? ELLC_OK : main_waits_batches(h);
    if (rc) return rc;
    rc = stage_h2d_on(h, st, d_slots, slots, (size_t)n * sizeof(int));
    if (rc) return rc;
    h->launches += launch_pyramid(st, h->kf_img, h->geo.img_off[kLevels], d_slots, n, h->geo);
    h->launches += launch_select(st, h->kf_depth, h->kf_var, h->geo.win_off[kLevels], h->kf_img,
                                 h->geo.img_off[kLevels], h->kf_mask, h->kf_rowcount, h->kf_rowoff, h->kf_count,
                                 h->kf_geo, h->kf_pix, h->kf_ikf, h->K, d_slots, n, h->geo);
    CU_TRY(h, cudaGetLastError());
    for (int i = 0; i < n; ++i) h->kf_state[slots[i]] = 2;
    return ELLC_OK;
}

// Slots that were uploaded since the last call are prepared (pyramid, texels, selection) before anything reads them.  When the
// uploads are still in flight on the copy stream -- a caller that uploads batch k+1 while batch k is tracking -- the
// preparation goes to its own stream behind the uploads, so that it overlaps the tracking kernels of batch k (and fills the
// SMs its last wave leaves idle) instead of queueing behind them; the compute stream then waits for the preparation only.
// Safe: an upload already waits for every batch that reads its slot (guard_slot_write), and the preparation follows the upload.
static int flush_dirty(ellc_handle* h) {
    const bool side = h->uploads_pending && h->batch_seq > h->batch_done_seq;      // something may still be tracking
    if (h->uploads_pending) {                              // copy_stream is in order: the last upload's event covers them all
        CU_TRY(h, cudaStreamWaitEvent(side ? h->prep_stream : h->stream, h->up_ev, 0));
        h->uploads_pending = false;
    }
    if (h->hyp_pending) {                                  // depth / variance pyramids a hypothesis upload is still building on the main stream
        if (side) CU_TRY(h, cudaStreamWaitEvent(h->prep_stream, h->hyp_ev, 0));
        h->hyp_pending = false;
    }
    if (!h->fr_dirty.empty()) {
        std::vector<int> s;
        for (int v : h->fr_dirty) if (h->fr_state[v] == 1) { s.push_back(v); h->fr_state[v] = 3; }
        for (int v : s) h->fr_state[v] = 1;
        h->fr_dirty.clear();
        int rc = prepare_frames_impl(h, (int)s.size(), s.data(), side);
        if (rc) return rc;
    }
    if (!h->kf_dirty.empty()) {
        std::vector<int> s;
        for (int v : h->kf_dirty) if (h->kf_state[v] == 1) { s.push_back(v); h->kf_state[v] = 3; }
        for (int v : s) h->kf_state[v] = 1;
        h->kf_dirty.clear();
        int rc = prepare_keyframes_impl(h, (int)s.size(), s.data(), side);
        if (rc) return rc;
    }
    if (side) {                                            // also orders the compute stream behind the uploads themselves
        CU_TRY(h, cudaEventRecord(h->prep_ev, h->prep_stream));
        CU_TRY(h, cudaStreamWaitEvent(h->stream, h->prep_ev, 0));
    }
    return ELLC_OK;
}

// Pools of the constant-weight loop-closure path: frame weight images (display_weightimg of ELLC_PAIR_SAVE_WEIGHTS tracks),
// keyframe weight pyramids, loop-closure records and hessians.  ~3 x the selection-list memory, so only on first use.
static int ensure_lc_pools(ellc_handle* h) {
    if (h->kf_weight) return ELLC_OK;
    const int64_t win = h->geo.win_off[kLevels];
    const int64_t nf = h->cfg.max_frames, nk = h->cfg.max_keyframes;
    CU_TRY(h, cudaMalloc(&h->fr_weight, (size_t)(nf * win) * sizeof(float)));
    CU_TRY(h, cudaMalloc(&h->kf_lc, (size_t)(nk * win + kRecTail) * sizeof(LcRec)));
    CU_TRY(h, cudaMalloc(&h->kf_lcH, (size_t)nk * kLevels * kLcHStride * sizeof(float)));
    CU_TRY(h, cudaMalloc(&h->kf_weight, (size_t)(nk * win) * sizeof(float)));
    CU_TRY(h, cudaMemsetAsync(h->fr_weight, 0, (size_t)(nf * win) * sizeof(float), h->stream));
    CU_TRY(h, cudaMemsetAsync(h->kf_weight, 0, (size_t)(nk * win) * sizeof(float), h->stream));     // Mat::zeros, src/Frame.cpp:114-117
    CU_TRY(h, cudaMemsetAsync(h->kf_lc, 0, (size_t)(nk * win + kRecTail) * sizeof(LcRec), h->stream));
    CU_TRY(h, cudaMalloc(&h->kf_lcf, (size_t)(nk * win + kRecTail) * sizeof(float4)));
    CU_TRY(h, cudaMalloc(&h->kf_lcp, (size_t)(nk * win + kRecTail) * sizeof(uint32_t)));
    CU_TRY(h, cudaMemsetAsync(h->kf_lcf, 0, (size_t)(nk * win + kRecTail) * sizeof(float4), h->stream));
    CU_TRY(h, cudaMemsetAsync(h->kf_lcp, 0, (size_t)(nk * win + kRecTail) * sizeof(uint32_t), h->stream));
    return ELLC_OK;
}

static void fill_params(const ellc_handle* h, TrackParams& p) {
    std::memset(&p, 0, sizeof(p));
    p.geo = h->geo;
    for (int l = 0; l < kLevels; ++l) { p.K[l] = h->K[l]; p.max_iter[l] = h->cfg.max_iter[l]; }
    p.huber_half = h->cfg.huber_d / 2;
    p.noise2 = h->cfg.camera_pixel_noise_2;
    for (int i = 0; i < 6; ++i) p.weight[i] = h->cfg.weight[i];
    p.stop_threshold = h->cfg.stop_threshold;
    p.jacobian_at_warped = h->cfg.jacobian_at_warped;
    p.tex_pool = h->fr_tex; p.tex_slot_stride = h->geo.win_off[kLevels] + kTexPad;
    p.geo_pool = h->kf_geo; p.pix_pool = h->kf_pix; p.ikf_pool = h->kf_ikf; p.rec_slot_stride = h->geo.win_off[kLevels];
    p.count_pool = h->kf_count;
    p.frw_pool = h->fr_weight; p.lc_pool = h->kf_lc; p.lc_H = h->kf_lcH; p.lcf_pool = h->kf_lcf; p.lcp_pool = h->kf_lcp;
    p.level_hi = kLevels - 1; p.level_lo = 0;
    p.pairs_per_cta = 1;
    p.lm_lambda = h->cfg.lm_lambda > 0.f ? h->cfg.lm_lambda : 0.f;
    p.lm_up = h->cfg.lm_up > 1.f ? h->cfg.lm_up : 4.0f;
    p.lm_down = (h->cfg.lm_down > 0.f && h->cfg.lm_down <= 1.f) ? h->cfg.lm_down : 0.5f;
    p.rowoff_pool = h->kf_rowoff; p.rows_total = h->rows_total; p.lc_bands = h->cfg.lc_bands;
}

static int pick_cluster(const ellc_handle* h, int n) {
    if (h->cfg.arithmetic == ELLC_ARITH_REFERENCE) return 1;
    int c = h->cfg.ctas_per_pair;
    if (c == 1 || c == 2 || c == 4 || c == 8) return c;
    if (n >= 148) return 1;
    c = 8;
    while (c > 1 && (int64_t)n * c > 296) c >>= 1;
    return c;
}

// Pairs per CTA (lockstep slots): with enough pairs to fill the GPU several times over, two pairs per CTA overlap their
// serial solves; small batches keep one pair per CTA so that every SM gets work.
static int pick_pairs_per_cta(const ellc_handle* h, int n, int cluster) {
    if (cluster != 1 || h->cfg.arithmetic == ELLC_ARITH_REFERENCE) return 1;
    int np = h->cfg.pairs_per_cta;
    if (const char* e = std::getenv("ELLC_PAIRS_PER_CTA")) np = std::atoi(e);
    if (np >= 1 && np <= 4) return np;
    return 1;                                              // measured: 2 is within noise of 1 (the other CTA of the SM already fills the solve gap)
}

static int validate_pairs(ellc_handle* h, int n, const ellc_pair* pairs) {
    for (int i = 0; i < n; ++i) {
        const ellc_pair& q = pairs[i];
        if (q.kf_slot < 0 || q.kf_slot >= h->cfg.max_keyframes || q.frame_slot < 0 || q.frame_slot >= h->cfg.max_frames) {
            h->err = "pair references a slot out of range";
            return ELLC_ERR_INVALID;
        }
        if (h->kf_state[q.kf_slot] == 0 || h->fr_state[q.frame_slot] == 0) {
            h->err = "pair references a slot that was never uploaded";
            return ELLC_ERR_NOT_READY;
        }
        if ((q.flags & ELLC_PAIR_CONST_WEIGHT) && (q.flags & ELLC_PAIR_SAVE_WEIGHTS)) {
            h->err = "a pair cannot both use constant weights and save weights (src/ImageFunc.cpp:241, :280)";
            return ELLC_ERR_INVALID;
        }
        if ((q.flags & ELLC_PAIR_CONST_WEIGHT) && !h->kf_lc_ready[q.kf_slot]) {
            h->err = "constant-weight pair on a keyframe without loop-closure records: call ellc_prepare_keyframes_lc after the keyframe's last upload";
            return ELLC_ERR_NOT_READY;
        }
    }
    return ELLC_OK;
}

static int xchg_publish(ellc_handle* h, cudaStream_t st) {
    ellc_exchange* xc = h->xc;
    if (!xc || !xc->attached || xc->consumed <= xc->published) return ELLC_OK;
    h->launches += launch_xchg_store(st, &reinterpret_cast<XchgHeader*>(xc->block)->released[0], (unsigned long long)xc->consumed);
    CU_TRY(h, cudaGetLastError());
    xc->published = xc->consumed;
    return ELLC_OK;
}

// Bookkeeping every tracking call shares (ellc_track_batch*, ellc_track_sequence_steps).  batch_begin numbers the batch; its
// completion event batch_ev[seq & 3] and timing events ev0r / ev1r are those of batch seq - 4, which is waited for first (ring of
// 4).
static int batch_begin(ellc_handle* h, long long* seq_out) {
    const long long seq = h->batch_seq + 1;
    if (seq > 4 && seq - 4 > h->batch_done_seq) {
        CU_TRY(h, cudaEventSynchronize(h->batch_ev[seq & 3]));
        if (seq - 4 > h->batch_done_seq) h->batch_done_seq = seq - 4;          // batches complete in order of their streams' events
    }
    *seq_out = seq;
    return ELLC_OK;
}
// Ordering of the batch's stream: behind everything enqueued on the main stream so far (synchronous preparation, weight
// and loop-closure kernels, and -- through the main stream's wait on prep_ev -- the pipelined preparation); NOT behind the
// previous batch, which runs on the other tracking stream, unless this batch shares buffers with it (serial: trace, weight images).
static int batch_order(ellc_handle* h, long long seq, bool serial) {
    cudaStream_t ts = h->tstream[seq & 1];
    CU_TRY(h, cudaEventRecord(h->main_ev, h->stream));
    CU_TRY(h, cudaStreamWaitEvent(ts, h->main_ev, 0));
    if (serial && seq > 1 && seq - 1 > h->batch_done_seq) CU_TRY(h, cudaStreamWaitEvent(ts, h->batch_ev[(seq - 1) & 3], 0));
    return xchg_publish(h, ts);                            // tables this rank has copied out since its last batch: tell the senders
}
// The batch's kernels are enqueued: its completion event, after which it is the last batch
static int batch_end(ellc_handle* h, long long seq) {
    cudaStream_t ts = h->tstream[seq & 1];
    CU_TRY(h, cudaEventRecord(h->ev1r[seq & 3], ts));
    CU_TRY(h, cudaEventRecord(h->batch_ev[seq & 3], ts));
    h->batch_seq = seq;
    return ELLC_OK;
}

// Launch parameters of the optional result exchange of a batch (ellc_track_batch_exchange)
struct XchgLaunch {
    int n_dst = 0;
    ellc_result* dst[ELLC_MAX_RANKS] = {};
    const int32_t* global_index = nullptr;                 // host
};

// A pair list that already lives on the device (ellc_lc_generate_pairs): no staging, no host-side schedule
struct DevicePairs {
    const ellc_pair* d_pairs;
    int flags;                                             // the same ELLC_PAIR_* flags on every pair
    const std::vector<int>* kf_slots;
    const std::vector<int>* frame_slots;
};

static int track_launch(ellc_handle* h, int n, const ellc_pair* pairs, bool want_trace, const XchgLaunch* xl = nullptr,
                        const DevicePairs* dev = nullptr) {
    int rc = dev ? ELLC_OK : validate_pairs(h, n, pairs);
    if (rc) return rc;
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    rc = flush_dirty(h);
    if (rc) return rc;
    // batch bookkeeping: sequence number, ring entry (staging + result buffers: a finished batch can be downloaded while the next two
    // run), completion event
    long long seq = 0;
    rc = batch_begin(h, &seq);
    if (rc) return rc;
    const int r = (int)(seq & 3);
    rc = ensure_ring_cap(h, r, n, want_trace);
    if (rc) return rc;
    h->d_pairs = h->d_pairs4[r]; h->d_order = h->d_order4[r]; h->d_results = h->d_results4[r];
    cudaStream_t ts = h->tstream[seq & 1];
    // Schedule: frame-major, keyframe-minor.  Pairs are independent, so the order is free; putting the K pairs of one
    // frame on adjacent CTAs makes them share that frame's texel pyramid in L2 (and, with few keyframes, the keyframe
    // selection lists stay L2-resident as well).  Results are still written at the caller's pair index.
    // Constant-weight (loop-closure) pairs run in their own kernel: the schedule lists the forward pairs first.
    int n_fwd = 0;
    bool save_weights = false;
    std::vector<int> order(dev ? 0 : n);
    if (dev) {                                             // generated lists are query-major = frame-major already
        n_fwd = (dev->flags & ELLC_PAIR_CONST_WEIGHT) ? 0 : n;
        save_weights = (dev->flags & ELLC_PAIR_SAVE_WEIGHTS) != 0;
    } else {
        for (int i = 0; i < n; ++i) order[i] = i;
        int kf_group = 0;                                  // EXPERIMENT: keyframes per schedule group (0 = frame-major over all keyframes)
        if (const char* e = std::getenv("ELLC_ORDER_KF_GROUP")) kf_group = std::atoi(e);
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
            const int la = (pairs[a].flags & ELLC_PAIR_CONST_WEIGHT) ? 1 : 0, lb = (pairs[b].flags & ELLC_PAIR_CONST_WEIGHT) ? 1 : 0;
            if (la != lb) return la < lb;
            if (kf_group > 0) {
                const int ga = pairs[a].kf_slot / kf_group, gb = pairs[b].kf_slot / kf_group;
                if (ga != gb) return ga < gb;
            }
            if (pairs[a].frame_slot != pairs[b].frame_slot) return pairs[a].frame_slot < pairs[b].frame_slot;
            return pairs[a].kf_slot < pairs[b].kf_slot;
        });
        for (int i = 0; i < n; ++i) {
            if (!(pairs[i].flags & ELLC_PAIR_CONST_WEIGHT)) ++n_fwd;
            if (pairs[i].flags & ELLC_PAIR_SAVE_WEIGHTS) save_weights = true;
        }
    }
    if (save_weights || n_fwd < n) {
        rc = ensure_lc_pools(h);
        if (rc) return rc;
    }
    rc = batch_order(h, seq, !h->overlap_batches || want_trace || save_weights || n_fwd < n);
    if (rc) return rc;
    if (!dev) {
        rc = stage_h2d_on(h, ts, h->d_pairs, pairs, (size_t)n * sizeof(ellc_pair));
        if (rc) return rc;
        rc = stage_h2d_on(h, ts, h->d_order, order.data(), (size_t)n * sizeof(int));
        if (rc) return rc;
    }
    if (xl && xl->n_dst > 0) {
        rc = stage_h2d_on(h, ts, h->d_gidx4[r], xl->global_index, (size_t)n * sizeof(int));
        if (rc) return rc;
    }
    if (want_trace) CU_TRY(h, cudaMemsetAsync(h->d_trace, 0, (size_t)n * kLevels * ELLC_MAX_TRACE_ITERS * sizeof(ellc_iter_trace), ts));
    TrackParams p;
    fill_params(h, p);
    p.pairs = dev ? dev->d_pairs : h->d_pairs; p.order = dev ? nullptr : h->d_order; p.results = h->d_results;
    p.trace = want_trace ? h->d_trace : nullptr; p.n_pairs = n;
    if (xl && xl->n_dst > 0) {
        p.xchg_n = xl->n_dst;
        for (int d = 0; d < xl->n_dst; ++d) p.xchg_dst[d] = xl->dst[d];
        p.xchg_index = h->d_gidx4[r];
    }
    CU_TRY(h, cudaEventRecord(h->ev0r[r], ts));
    p.n_pairs = n_fwd;
    const int cluster = pick_cluster(h, n_fwd);
    p.pairs_per_cta = pick_pairs_per_cta(h, n_fwd, cluster);
    // diagnostics (tools/gpu_solve_cost.sh): fixed iteration counts with / without the solve
    if (const char* e = std::getenv("ELLC_DEBUG_NO_UPDATE")) if (*e == '1') p.no_update = 1;
    if (const char* e = std::getenv("ELLC_DEBUG_MAX_ITER")) std::sscanf(e, "%d,%d,%d,%d", &p.max_iter[0], &p.max_iter[1], &p.max_iter[2], &p.max_iter[3]);
    if (const char* e = std::getenv("ELLC_DEBUG_NO_STOP")) if (*e == '1') p.stop_threshold = -1.0f;
    // Scheduling of the forward pairs: a cluster of CTAs per pair (few pairs: latency) or one CTA per 1..4 lockstep pairs
    int l = launch_track(ts, p, cluster, h->cfg.arithmetic);
    if (l < 0) { h->err = std::string("track kernel launch failed: ") + cudaGetErrorString(cudaGetLastError()); return ELLC_ERR_CUDA; }
    h->launches += l;
    if (n_fwd < n) {
        p.order = dev ? nullptr : h->d_order + n_fwd;
        p.n_pairs = n - n_fwd;
        l = launch_track_lc(ts, p, h->cfg.arithmetic);
        if (l < 0) { h->err = std::string("loop-closure track kernel launch failed: ") + cudaGetErrorString(cudaGetLastError()); return ELLC_ERR_CUDA; }
        h->launches += l;
    }
    rc = batch_end(h, seq);
    if (rc) return rc;
    h->res_seq[r] = seq;
    h->res_taken[r] = xl != nullptr;                       // exchanged batches are read from the exchange tables, not from this buffer
    if (dev) {
        for (int v : *dev->frame_slots) h->fr_reader[v] = seq;
        for (int v : *dev->kf_slots) h->kf_reader[v] = seq;
    } else {
        for (int i = 0; i < n; ++i) { h->fr_reader[pairs[i].frame_slot] = seq; h->kf_reader[pairs[i].kf_slot] = seq; }
    }
    CU_TRY(h, cudaGetLastError());
    return ELLC_OK;
}

extern "C" {

int ellc_upload_frame(ellc_handle* h, int32_t slot, const uint8_t* image) {
    if (!h) return ELLC_ERR_INVALID;
    if (!image || slot < 0 || slot >= h->cfg.max_frames) { h->err = "bad frame slot / null image"; return ELLC_ERR_INVALID; }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = guard_slot_write(h, h->fr_reader[slot]);
    if (rc) return rc;
    CU_TRY(h, cudaMemcpyAsync(h->fr_img + (int64_t)slot * h->geo.img_off[kLevels], image, (size_t)h->geo.img_off[1],
                              cudaMemcpyHostToDevice, h->copy_stream));
    h->fr_state[slot] = 1;
    h->fr_hist_ready[slot] = 0;
    h->fr_dirty.push_back(slot);
    return after_upload(h);
}

int ellc_upload_keyframe(ellc_handle* h, int32_t slot, const uint8_t* image, const float* const depth[ELLC_LEVELS],
                         const float* const var[ELLC_LEVELS]) {
    if (!h) return ELLC_ERR_INVALID;
    if (!image || !depth || !var || slot < 0 || slot >= h->cfg.max_keyframes) { h->err = "bad keyframe slot / null pointer"; return ELLC_ERR_INVALID; }
    for (int l = 0; l < kLevels; ++l) if (!depth[l] || !var[l]) { h->err = "null depth/var level"; return ELLC_ERR_INVALID; }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = guard_slot_write(h, h->kf_reader[slot]);
    if (rc) return rc;
    CU_TRY(h, cudaMemcpyAsync(h->kf_img + (int64_t)slot * h->geo.img_off[kLevels], image, (size_t)h->geo.img_off[1],
                              cudaMemcpyHostToDevice, h->copy_stream));
    const int64_t win = h->geo.win_off[kLevels];
    for (int l = 0; l < kLevels; ++l) {
        const size_t bytes = (size_t)(h->geo.win_off[l + 1] - h->geo.win_off[l]) * sizeof(float);
        CU_TRY(h, cudaMemcpyAsync(h->kf_depth + slot * win + h->geo.win_off[l], depth[l], bytes, cudaMemcpyHostToDevice, h->copy_stream));
        CU_TRY(h, cudaMemcpyAsync(h->kf_var + slot * win + h->geo.win_off[l], var[l], bytes, cudaMemcpyHostToDevice, h->copy_stream));
    }
    h->kf_state[slot] = 1;
    h->kf_lc_ready[slot] = 0;                              // the loop-closure records describe the previous contents
    h->kf_nvalid[slot] = -1;
    h->kf_dirty.push_back(slot);
    return after_upload(h);
}

int ellc_set_camera(ellc_handle* h, const ellc_camera* cam) {
    if (!h) return ELLC_ERR_INVALID;
    if (!cam) { h->err = "null camera"; return ELLC_ERR_INVALID; }
    const int W = h->cfg.width, H = h->cfg.height;
    if ((cam->channels != 1 && cam->channels != 3) || (cam->undistort != 0 && cam->undistort != 1) || cam->width < W || cam->height < H ||
        cam->width > 16384 || cam->height > 16384 || (int64_t)cam->pitch < (int64_t)cam->width * cam->channels) {
        h->err = "unsupported camera (channels 1 or 3, undistort 0 or 1, working size <= camera size <= 16384, pitch >= width * channels)";
        return ELLC_ERR_INVALID;
    }
    UndistortParams up;
    std::memset(&up, 0, sizeof(up));
    if (cam->undistort) {
        for (int i = 0; i < 9; ++i) if (!std::isfinite(cam->K[i]) || !std::isfinite(cam->new_K[i])) { h->err = "non-finite camera matrix"; return ELLC_ERR_INVALID; }
        for (int i = 0; i < 5; ++i) if (!std::isfinite(cam->dist[i])) { h->err = "non-finite distortion coefficient"; return ELLC_ERR_INVALID; }
        if (!invert3(cam->new_K, up.ir)) { h->err = "singular new_K"; return ELLC_ERR_INVALID; }
        up.fx = cam->K[0]; up.fy = cam->K[4]; up.u0 = cam->K[2]; up.v0 = cam->K[5];
        up.k1 = cam->dist[0]; up.k2 = cam->dist[1]; up.p1 = cam->dist[2]; up.p2 = cam->dist[3]; up.k3 = cam->dist[4];
    }
    std::vector<int4> cols(W), rows(H);
    build_resize_taps(cam->width, cam->height, W, H, cols.data(), rows.data());
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    // the tables are read by ingestion kernels only (preparation stream), whose inputs come through the copy stream
    CU_TRY(h, cudaStreamSynchronize(h->copy_stream));
    CU_TRY(h, cudaStreamSynchronize(h->prep_stream));
    if (!h->d_cam_cols) {
        CU_TRY(h, cudaMalloc(&h->d_cam_cols, (size_t)W * sizeof(int4)));
        CU_TRY(h, cudaMalloc(&h->d_cam_rows, (size_t)H * sizeof(int4)));
        CU_TRY(h, cudaMalloc(&h->d_cam_map, (size_t)4 * W * H * sizeof(uint2)));
        CU_TRY(h, cudaMalloc(&h->d_ingest_jobs, (size_t)h->slots_cap * sizeof(IngestJob)));
    }
    IngestGeo g = {cam->width, cam->height, cam->channels, cam->pitch, W, H, cam->undistort, 0};
    CU_TRY(h, cudaMemcpyAsync(h->d_cam_cols, cols.data(), (size_t)W * sizeof(int4), cudaMemcpyHostToDevice, h->prep_stream));
    CU_TRY(h, cudaMemcpyAsync(h->d_cam_rows, rows.data(), (size_t)H * sizeof(int4), cudaMemcpyHostToDevice, h->prep_stream));
    if (cam->undistort) h->launches += launch_undistort_map(h->prep_stream, g, up, h->d_cam_cols, h->d_cam_rows, h->d_cam_map);
    else CU_TRY(h, cudaMemsetAsync(h->d_cam_map, 0, (size_t)4 * W * H * sizeof(uint2), h->prep_stream));
    CU_TRY(h, cudaGetLastError());
    CU_TRY(h, cudaStreamSynchronize(h->prep_stream));       // cols / rows are host temporaries
    h->cam_geo = g;
    h->cam_set = true;
    return ELLC_OK;
}

int ellc_read_camera_tables(ellc_handle* h, int32_t* tap_x, int32_t* tap_y, int16_t* map_xy, uint16_t* map_frac) {
    if (!h) return ELLC_ERR_INVALID;
    if (!h->cam_set) { h->err = "no camera set (ellc_set_camera)"; return ELLC_ERR_NOT_READY; }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    const int W = h->cfg.width, H = h->cfg.height;
    std::vector<int4> cols(W), rows(H);
    std::vector<uint2> map((size_t)4 * W * H);
    CU_TRY(h, cudaMemcpyAsync(cols.data(), h->d_cam_cols, (size_t)W * sizeof(int4), cudaMemcpyDeviceToHost, h->prep_stream));
    CU_TRY(h, cudaMemcpyAsync(rows.data(), h->d_cam_rows, (size_t)H * sizeof(int4), cudaMemcpyDeviceToHost, h->prep_stream));
    CU_TRY(h, cudaMemcpyAsync(map.data(), h->d_cam_map, map.size() * sizeof(uint2), cudaMemcpyDeviceToHost, h->prep_stream));
    CU_TRY(h, cudaStreamSynchronize(h->prep_stream));
    for (int i = 0; i < W; ++i) if (tap_x) { tap_x[2 * i] = cols[i].x; tap_x[2 * i + 1] = cols[i].y; }
    for (int i = 0; i < H; ++i) if (tap_y) { tap_y[2 * i] = rows[i].x; tap_y[2 * i + 1] = rows[i].y; }
    for (size_t i = 0; i < map.size(); ++i) {
        if (map_xy) { map_xy[2 * i] = (int16_t)(map[i].x & 0xffffu); map_xy[2 * i + 1] = (int16_t)(map[i].x >> 16); }
        if (map_frac) map_frac[i] = (uint16_t)map[i].y;
    }
    return ELLC_OK;
}

}  // extern "C"

// n camera images -> level-0 images of n distinct slots of one pool.  Chain: copy stream (waits for the batches that read the
// slots, guard_slot_write; copies host images into the staging buffer) -> ingest kernel on the preparation stream -> copy stream
// (so that every consumer that waits for uploads, and the next staging copy, waits for the kernel too).
static int ingest_impl(ellc_handle* h, int n, const int32_t* slots, const uint8_t* const* images, bool on_device, bool keyframe) {
    const IngestGeo& g = h->cam_geo;
    const size_t bytes = (size_t)g.pitch * (g.cam_h - 1) + (size_t)g.cam_w * g.channels, stride = (bytes + 255) & ~(size_t)255;
    for (int i = 0; i < n; ++i) {
        int rc = guard_slot_write(h, keyframe ? h->kf_reader[slots[i]] : h->fr_reader[slots[i]]);
        if (rc) return rc;
    }
    std::vector<IngestJob> jobs(n);
    uint8_t* pool = keyframe ? h->kf_img : h->fr_img;
    for (int i = 0; i < n; ++i) jobs[i].dst = pool + (int64_t)slots[i] * h->geo.img_off[kLevels];
    if (on_device) {
        for (int i = 0; i < n; ++i) jobs[i].src = images[i];
    } else {
        if ((size_t)n * stride > h->cam_stage_cap) {       // the previous ingestion kernels may still read the old buffer
            CU_TRY(h, cudaStreamSynchronize(h->copy_stream));
            CU_TRY(h, cudaStreamSynchronize(h->prep_stream));
            cudaFree(h->d_cam_stage); h->d_cam_stage = nullptr; h->cam_stage_cap = 0;
            CU_TRY(h, cudaMalloc(&h->d_cam_stage, (size_t)n * stride));
            h->cam_stage_cap = (size_t)n * stride;
        }
        for (int i = 0; i < n; ++i) {
            jobs[i].src = h->d_cam_stage + (size_t)i * stride;
            CU_TRY(h, cudaMemcpyAsync(h->d_cam_stage + (size_t)i * stride, images[i], bytes, cudaMemcpyHostToDevice, h->copy_stream));
        }
    }
    CU_TRY(h, cudaEventRecord(h->ingest_ev, h->copy_stream));
    CU_TRY(h, cudaStreamWaitEvent(h->prep_stream, h->ingest_ev, 0));
    int rc = stage_h2d_on(h, h->prep_stream, h->d_ingest_jobs, jobs.data(), (size_t)n * sizeof(IngestJob));
    if (rc) return rc;
    h->launches += launch_ingest(h->prep_stream, h->d_ingest_jobs, n, g, h->d_cam_cols, h->d_cam_rows, h->d_cam_map);
    CU_TRY(h, cudaGetLastError());
    CU_TRY(h, cudaEventRecord(h->ingest_ev, h->prep_stream));
    CU_TRY(h, cudaStreamWaitEvent(h->copy_stream, h->ingest_ev, 0));
    for (int i = 0; i < n; ++i) {
        const int s = slots[i];
        if (keyframe) { h->kf_state[s] = 1; h->kf_lc_ready[s] = 0; h->kf_nvalid[s] = -1; h->kf_dirty.push_back(s); }
        else { h->fr_state[s] = 1; h->fr_hist_ready[s] = 0; h->fr_dirty.push_back(s); }
    }
    return after_upload(h);
}

extern "C" {

int ellc_ingest_frames(ellc_handle* h, int32_t n, const int32_t* slots, const uint8_t* const* images, int32_t on_device) {
    if (!h) return ELLC_ERR_INVALID;
    if (n < 0 || n > h->cfg.max_frames || (n > 0 && (!slots || !images)) || (on_device != 0 && on_device != 1)) {
        h->err = "bad frame slot list / image list"; return ELLC_ERR_INVALID;
    }
    std::vector<char> seen(h->cfg.max_frames, 0);
    for (int i = 0; i < n; ++i) {
        if (slots[i] < 0 || slots[i] >= h->cfg.max_frames || seen[slots[i]] || !images[i]) { h->err = "frame slot out of range / repeated, or null image"; return ELLC_ERR_INVALID; }
        seen[slots[i]] = 1;
    }
    if (!h->cam_set) { h->err = "no camera set (ellc_set_camera)"; return ELLC_ERR_NOT_READY; }
    if (n == 0) return ELLC_OK;
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    return ingest_impl(h, n, slots, images, on_device == 1, false);
}

int ellc_ingest_keyframe(ellc_handle* h, int32_t slot, const uint8_t* image, int32_t on_device, const float* const depth[ELLC_LEVELS],
                         const float* const var[ELLC_LEVELS]) {
    if (!h) return ELLC_ERR_INVALID;
    if (!image || !depth || !var || slot < 0 || slot >= h->cfg.max_keyframes || (on_device != 0 && on_device != 1)) { h->err = "bad keyframe slot / null pointer"; return ELLC_ERR_INVALID; }
    for (int l = 0; l < kLevels; ++l) if (!depth[l] || !var[l]) { h->err = "null depth/var level"; return ELLC_ERR_INVALID; }
    if (!h->cam_set) { h->err = "no camera set (ellc_set_camera)"; return ELLC_ERR_NOT_READY; }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = guard_slot_write(h, h->kf_reader[slot]);
    if (rc) return rc;
    const int64_t win = h->geo.win_off[kLevels];
    for (int l = 0; l < kLevels; ++l) {
        const size_t bytes = (size_t)(h->geo.win_off[l + 1] - h->geo.win_off[l]) * sizeof(float);
        CU_TRY(h, cudaMemcpyAsync(h->kf_depth + slot * win + h->geo.win_off[l], depth[l], bytes, cudaMemcpyHostToDevice, h->copy_stream));
        CU_TRY(h, cudaMemcpyAsync(h->kf_var + slot * win + h->geo.win_off[l], var[l], bytes, cudaMemcpyHostToDevice, h->copy_stream));
    }
    return ingest_impl(h, 1, &slot, &image, on_device == 1, true);
}

int ellc_upload_keyframe_hypotheses(ellc_handle* h, int32_t slot, const uint8_t* image, const uint8_t* valid,
                                    const float* inv_depth_smoothed, const float* variance_smoothed, uint8_t* valid_out) {
    if (!h) return ELLC_ERR_INVALID;
    if (!image || !valid || !inv_depth_smoothed || !variance_smoothed || slot < 0 || slot >= h->cfg.max_keyframes) {
        h->err = "bad keyframe slot / null pointer"; return ELLC_ERR_INVALID;
    }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    const int64_t npx = (int64_t)h->geo.width * h->geo.height, win = h->geo.win_off[kLevels];
    if (!h->d_hyp) {
        CU_TRY(h, cudaMalloc(&h->d_hyp, (size_t)npx * 10));                  // valid u8 | idepth f32 | var f32 | valid_out u8
        CU_TRY(h, cudaMalloc(&h->d_nvalid, (size_t)h->cfg.max_keyframes * sizeof(int)));
    }
    int rc = guard_slot_write(h, h->kf_reader[slot]);
    if (rc) return rc;
    // the staging buffer is shared by all slots: the previous call's kernels (compute stream) must be done with it
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    uint8_t* d_valid = h->d_hyp + 8 * npx;
    float* d_idepth = reinterpret_cast<float*>(h->d_hyp);
    float* d_vars = d_idepth + npx;
    uint8_t* d_vout = d_valid + npx;
    CU_TRY(h, cudaMemcpyAsync(h->kf_img + (int64_t)slot * h->geo.img_off[kLevels], image, (size_t)h->geo.img_off[1], cudaMemcpyHostToDevice, h->copy_stream));
    CU_TRY(h, cudaMemcpyAsync(d_valid, valid, (size_t)npx, cudaMemcpyHostToDevice, h->copy_stream));
    CU_TRY(h, cudaMemcpyAsync(d_idepth, inv_depth_smoothed, (size_t)npx * 4, cudaMemcpyHostToDevice, h->copy_stream));
    CU_TRY(h, cudaMemcpyAsync(d_vars, variance_smoothed, (size_t)npx * 4, cudaMemcpyHostToDevice, h->copy_stream));
    rc = after_upload(h);
    if (rc) return rc;
    CU_TRY(h, cudaStreamWaitEvent(h->stream, h->up_ev, 0));
    rc = main_waits_batches(h);                            // a batch in flight may still read this slot's depth / variance
    if (rc) return rc;
    CU_TRY(h, cudaMemsetAsync(h->d_nvalid + slot, 0, sizeof(int), h->stream));
    h->launches += launch_depth_pyramid(h->stream, d_valid, d_idepth, d_vars, h->kf_depth + slot * win, h->kf_var + slot * win,
                                        valid_out ? d_vout : nullptr, h->d_nvalid + slot, h->geo);
    CU_TRY(h, cudaGetLastError());
    // the pipelined preparation (flush_dirty's side path, ellc_prepare_async) runs on its own stream: it must see these pyramids
    CU_TRY(h, cudaEventRecord(h->hyp_ev, h->stream));
    h->hyp_pending = true;
    if (valid_out) {
        CU_TRY(h, cudaMemcpyAsync(valid_out, d_vout, (size_t)npx, cudaMemcpyDeviceToHost, h->stream));
        CU_TRY(h, cudaStreamSynchronize(h->stream));
    }
    h->kf_nvalid[slot] = -2;                               // on the device, not fetched yet
    h->kf_state[slot] = 1;
    h->kf_lc_ready[slot] = 0;
    h->kf_dirty.push_back(slot);
    return ELLC_OK;
}

int ellc_read_keyframe_occupancy(ellc_handle* h, int32_t slot, int32_t* n_valid, float* occupancy) {
    if (!h) return ELLC_ERR_INVALID;
    if (slot < 0 || slot >= h->cfg.max_keyframes) { h->err = "bad keyframe slot"; return ELLC_ERR_INVALID; }
    if (h->kf_nvalid[slot] == -1) { h->err = "keyframe slot was not uploaded from hypotheses"; return ELLC_ERR_NOT_READY; }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    if (h->kf_nvalid[slot] == -2) {
        int v = 0;
        CU_TRY(h, cudaMemcpyAsync(&v, h->d_nvalid + slot, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CU_TRY(h, cudaStreamSynchronize(h->stream));
        h->kf_nvalid[slot] = v;
    }
    if (n_valid) *n_valid = h->kf_nvalid[slot];
    // depthMap::calculate_no_of_Seeds, src/DepthPropagation.cpp:1804-1830: float count / int(W*H) * 100
    if (occupancy) *occupancy = (float)h->kf_nvalid[slot] / (h->geo.width * h->geo.height) * 100;
    return ELLC_OK;
}

int ellc_read_keyframe_depth(ellc_handle* h, int32_t slot, int32_t level, float* depth, float* var) {
    if (!h) return ELLC_ERR_INVALID;
    if (slot < 0 || slot >= h->cfg.max_keyframes || level < 0 || level >= kLevels) { h->err = "bad slot/level"; return ELLC_ERR_INVALID; }
    if (h->kf_state[slot] == 0) { h->err = "keyframe slot empty"; return ELLC_ERR_NOT_READY; }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    CU_TRY(h, cudaStreamSynchronize(h->copy_stream));
    { int rcw = main_waits_batches(h); if (rcw) return rcw; }
    const int64_t win = h->geo.win_off[kLevels];
    const size_t bytes = (size_t)(h->geo.win_off[level + 1] - h->geo.win_off[level]) * sizeof(float);
    if (depth) CU_TRY(h, cudaMemcpyAsync(depth, h->kf_depth + slot * win + h->geo.win_off[level], bytes, cudaMemcpyDeviceToHost, h->stream));
    if (var) CU_TRY(h, cudaMemcpyAsync(var, h->kf_var + slot * win + h->geo.win_off[level], bytes, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return ELLC_OK;
}

int ellc_frame_histograms(ellc_handle* h, int32_t n, const int32_t* frame_slots, float* hist) {
    if (!h) return ELLC_ERR_INVALID;
    if (n < 0 || (n > 0 && !frame_slots) || n > h->slots_cap) { h->err = "bad frame slot list"; return ELLC_ERR_INVALID; }
    for (int i = 0; i < n; ++i) {
        if (frame_slots[i] < 0 || frame_slots[i] >= h->cfg.max_frames) { h->err = "frame slot out of range"; return ELLC_ERR_INVALID; }
        if (h->fr_state[frame_slots[i]] == 0) { h->err = "frame slot empty"; return ELLC_ERR_NOT_READY; }
    }
    if (n == 0) return ELLC_OK;
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    if (!h->fr_hist) CU_TRY(h, cudaMalloc(&h->fr_hist, (size_t)h->cfg.max_frames * 256 * sizeof(float)));
    if (h->uploads_pending) { CU_TRY(h, cudaStreamWaitEvent(h->stream, h->up_ev, 0)); }      // the level-0 images must have landed
    int rc = stage_h2d(h, h->d_slots, frame_slots, (size_t)n * sizeof(int));
    if (rc) return rc;
    h->launches += launch_frame_histograms(h->stream, h->fr_img, h->geo.img_off[kLevels], h->d_slots, n, h->geo.width * h->geo.height, h->fr_hist);
    CU_TRY(h, cudaGetLastError());
    for (int i = 0; i < n; ++i) h->fr_hist_ready[frame_slots[i]] = 1;
    if (hist) {
        for (int i = 0; i < n; ++i)
            CU_TRY(h, cudaMemcpyAsync(hist + (size_t)i * 256, h->fr_hist + (size_t)frame_slots[i] * 256, 256 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
        CU_TRY(h, cudaStreamSynchronize(h->stream));
    }
    return ELLC_OK;
}

int ellc_lc_gate(ellc_handle* h, int32_t n, const ellc_lc_candidate* cand, float match_threshold, float max_rel_view_angle, ellc_lc_stats* stats) {
    if (!h) return ELLC_ERR_INVALID;
    if (n < 0 || (n > 0 && (!cand || !stats))) { h->err = "bad candidate list"; return ELLC_ERR_INVALID; }
    for (int i = 0; i < n; ++i) {
        const int a = cand[i].loop_frame_slot, b = cand[i].test_frame_slot;
        if (a < 0 || a >= h->cfg.max_frames || b < 0 || b >= h->cfg.max_frames) { h->err = "candidate frame slot out of range"; return ELLC_ERR_INVALID; }
        if (!h->fr_hist || !h->fr_hist_ready[a] || !h->fr_hist_ready[b]) { h->err = "candidate without histogram: call ellc_frame_histograms first"; return ELLC_ERR_NOT_READY; }
    }
    if (n == 0) return ELLC_OK;
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    const size_t in_bytes = (size_t)n * sizeof(ellc_lc_candidate), out_bytes = (size_t)n * sizeof(ellc_lc_stats);
    void* d_buf = nullptr;
    CU_TRY(h, cudaMallocAsync(&d_buf, in_bytes + out_bytes, h->stream));
    ellc_lc_candidate* d_cand = reinterpret_cast<ellc_lc_candidate*>(d_buf);
    ellc_lc_stats* d_out = reinterpret_cast<ellc_lc_stats*>(reinterpret_cast<char*>(d_buf) + in_bytes);
    CU_TRY(h, cudaMemcpyAsync(d_cand, cand, in_bytes, cudaMemcpyHostToDevice, h->stream));
    h->launches += launch_lc_gate(h->stream, h->fr_hist, d_cand, n, match_threshold, max_rel_view_angle, d_out);
    CU_TRY(h, cudaGetLastError());
    CU_TRY(h, cudaMemcpyAsync(stats, d_out, out_bytes, cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaFreeAsync(d_buf, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return ELLC_OK;
}

int ellc_lc_generate_pairs(ellc_handle* h, int32_t ring_len, const ellc_lc_ring_entry* ring, int32_t n_queries, const ellc_lc_query* queries,
                           int32_t min_match_difference, float match_threshold, float max_rel_view_angle, int32_t pair_flags,
                           int32_t* n_pairs, ellc_pair* pairs, ellc_lc_stats* stats, int32_t* query_of_pair) {
    if (!h) return ELLC_ERR_INVALID;
    if (ring_len < 1 || ring_len > 64 || n_queries < 0 || !ring || (n_queries > 0 && !queries) || !n_pairs) { h->err = "bad ring / query arguments (ring_len <= 64)"; return ELLC_ERR_INVALID; }
    if ((pair_flags & ELLC_PAIR_CONST_WEIGHT) && (pair_flags & ELLC_PAIR_SAVE_WEIGHTS)) { h->err = "a pair cannot both use constant weights and save weights"; return ELLC_ERR_INVALID; }
    *n_pairs = 0;
    h->gen_n = 0;
    h->gen_kf_slots.clear(); h->gen_frame_slots.clear();
    if (n_queries == 0) return ELLC_OK;
    for (int i = 0; i < ring_len; ++i) {
        if (!ring[i].is_valid) continue;
        const int fs = ring[i].frame_slot, ks = ring[i].kf_slot;
        if (fs < 0 || fs >= h->cfg.max_frames || ks < 0 || ks >= h->cfg.max_keyframes) { h->err = "ring entry references a slot out of range"; return ELLC_ERR_INVALID; }
        if (!h->fr_hist || !h->fr_hist_ready[fs]) { h->err = "ring entry without histogram: call ellc_frame_histograms first"; return ELLC_ERR_NOT_READY; }
        if (h->kf_state[ks] == 0) { h->err = "ring entry references a keyframe slot that was never uploaded"; return ELLC_ERR_NOT_READY; }
        if ((pair_flags & ELLC_PAIR_CONST_WEIGHT) && !h->kf_lc_ready[ks]) { h->err = "constant-weight pairs on a keyframe without loop-closure records"; return ELLC_ERR_NOT_READY; }
        h->gen_kf_slots.push_back(ks);
    }
    for (int q = 0; q < n_queries; ++q) {
        const int fs = queries[q].frame_slot;
        if (fs < 0 || fs >= h->cfg.max_frames || queries[q].current_array_id < 0 || queries[q].current_array_id > ring_len ||
            queries[q].match_window_beg < 0 || queries[q].match_window_beg >= ring_len || queries[q].match_window_end < 0 ||
            queries[q].match_window_end >= ring_len) { h->err = "query references a slot / ring position out of range"; return ELLC_ERR_INVALID; }
        if (h->fr_state[fs] == 0 || !h->fr_hist || !h->fr_hist_ready[fs]) { h->err = "query frame without histogram: call ellc_frame_histograms first"; return ELLC_ERR_NOT_READY; }
        h->gen_frame_slots.push_back(fs);
    }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = main_waits_batches(h);
    if (rc) return rc;
    const size_t cap = (size_t)n_queries * ring_len;
    auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const size_t o_ring = 0, o_q = o_ring + up((size_t)ring_len * sizeof(ellc_lc_ring_entry)), o_segp = o_q + up((size_t)n_queries * sizeof(ellc_lc_query)),
                 o_segs = o_segp + up(cap * sizeof(ellc_pair)), o_segc = o_segs + up(cap * sizeof(ellc_lc_stats)), o_p = o_segc + up((size_t)n_queries * sizeof(int)),
                 o_s = o_p + up(cap * sizeof(ellc_pair)), o_qi = o_s + up(cap * sizeof(ellc_lc_stats)), o_t = o_qi + up(cap * sizeof(int)), total = o_t + 256;
    if (total > h->gen_bytes) {
        CU_TRY(h, cudaStreamSynchronize(h->stream));
        for (int i = 0; i < 2; ++i) CU_TRY(h, cudaStreamSynchronize(h->tstream[i]));      // a batch may still read the previous list
        cudaFree(h->d_gen); h->d_gen = nullptr; h->gen_bytes = 0;
        CU_TRY(h, cudaMalloc(&h->d_gen, total));
        h->gen_bytes = total;
    }
    char* g = h->d_gen;
    rc = stage_h2d(h, g + o_ring, ring, (size_t)ring_len * sizeof(ellc_lc_ring_entry));
    if (rc) return rc;
    rc = stage_h2d(h, g + o_q, queries, (size_t)n_queries * sizeof(ellc_lc_query));
    if (rc) return rc;
    const int l = launch_lc_generate(h->stream, h->fr_hist, reinterpret_cast<ellc_lc_ring_entry*>(g + o_ring), ring_len, reinterpret_cast<ellc_lc_query*>(g + o_q),
                                     n_queries, min_match_difference, match_threshold, max_rel_view_angle, pair_flags, reinterpret_cast<ellc_pair*>(g + o_segp),
                                     reinterpret_cast<ellc_lc_stats*>(g + o_segs), reinterpret_cast<int*>(g + o_segc), reinterpret_cast<ellc_pair*>(g + o_p),
                                     reinterpret_cast<ellc_lc_stats*>(g + o_s), reinterpret_cast<int*>(g + o_qi), reinterpret_cast<int*>(g + o_t));
    if (l < 0) { h->err = "pair-list kernels: bad launch configuration"; return ELLC_ERR_INVALID; }
    h->launches += l;
    CU_TRY(h, cudaGetLastError());
    int n = 0;
    CU_TRY(h, cudaMemcpyAsync(&n, g + o_t, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    if (n > 0) {
        if (pairs) CU_TRY(h, cudaMemcpyAsync(pairs, g + o_p, (size_t)n * sizeof(ellc_pair), cudaMemcpyDeviceToHost, h->stream));
        if (stats) CU_TRY(h, cudaMemcpyAsync(stats, g + o_s, (size_t)n * sizeof(ellc_lc_stats), cudaMemcpyDeviceToHost, h->stream));
        if (query_of_pair) CU_TRY(h, cudaMemcpyAsync(query_of_pair, g + o_qi, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CU_TRY(h, cudaStreamSynchronize(h->stream));
    }
    h->d_gen_pairs = reinterpret_cast<ellc_pair*>(g + o_p);
    h->gen_n = n; h->gen_flags = pair_flags;
    *n_pairs = n;
    return ELLC_OK;
}

int ellc_track_generated_pairs(ellc_handle* h, int32_t n_pairs, ellc_result* results) {
    if (!h) return ELLC_ERR_INVALID;
    if (n_pairs < 0 || n_pairs != h->gen_n || (n_pairs > 0 && !results)) { h->err = "n_pairs is not what the last ellc_lc_generate_pairs reported / null results"; return ELLC_ERR_INVALID; }
    if (n_pairs == 0) return ELLC_OK;
    for (int ks : h->gen_kf_slots)
        if ((h->gen_flags & ELLC_PAIR_CONST_WEIGHT) && !h->kf_lc_ready[ks]) { h->err = "a keyframe of the generated list lost its loop-closure records"; return ELLC_ERR_NOT_READY; }
    DevicePairs dev = {h->d_gen_pairs, h->gen_flags, &h->gen_kf_slots, &h->gen_frame_slots};
    int rc = track_launch(h, n_pairs, nullptr, false, nullptr, &dev);
    if (rc) return rc;
    cudaStream_t ts = h->tstream[h->batch_seq & 1];
    CU_TRY(h, cudaMemcpyAsync(results, h->d_results, (size_t)n_pairs * sizeof(ellc_result), cudaMemcpyDeviceToHost, ts));
    CU_TRY(h, cudaStreamSynchronize(ts));
    note_done(h, h->batch_seq);
    return ELLC_OK;
}

int ellc_frame_image_devptr(ellc_handle* h, int32_t slot, uint8_t** image) {
    if (!h || !image || slot < 0 || slot >= h->cfg.max_frames) return ELLC_ERR_INVALID;
    *image = h->fr_img + (int64_t)slot * h->geo.img_off[kLevels];
    return ELLC_OK;
}

int ellc_keyframe_devptrs(ellc_handle* h, int32_t slot, uint8_t** image, float** depth, float** var,
                          int64_t level_offsets[ELLC_LEVELS + 1]) {
    if (!h || slot < 0 || slot >= h->cfg.max_keyframes) return ELLC_ERR_INVALID;
    const int64_t win = h->geo.win_off[kLevels];
    if (image) *image = h->kf_img + (int64_t)slot * h->geo.img_off[kLevels];
    if (depth) *depth = h->kf_depth + slot * win;
    if (var) *var = h->kf_var + slot * win;
    if (level_offsets) for (int l = 0; l <= kLevels; ++l) level_offsets[l] = h->geo.win_off[l];
    return ELLC_OK;
}

int ellc_prepare_frames(ellc_handle* h, int32_t n, const int32_t* slots) {
    if (!h || (n > 0 && !slots) || n > h->cfg.max_frames) return ELLC_ERR_INVALID;
    for (int i = 0; i < n; ++i) {
        if (slots[i] < 0 || slots[i] >= h->cfg.max_frames) { h->err = "frame slot out of range"; return ELLC_ERR_INVALID; }
        if (h->fr_state[slots[i]] == 0) { h->err = "frame slot empty"; return ELLC_ERR_NOT_READY; }
    }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    if (h->uploads_pending) CU_TRY(h, cudaStreamWaitEvent(h->stream, h->up_ev, 0));    // uploads run on the copy stream (the flag stays: other consumers wait too)
    return prepare_frames_impl(h, n, slots);
}

int ellc_prepare_keyframes(ellc_handle* h, int32_t n, const int32_t* slots) {
    if (!h || (n > 0 && !slots) || n > h->cfg.max_keyframes) return ELLC_ERR_INVALID;
    for (int i = 0; i < n; ++i) {
        if (slots[i] < 0 || slots[i] >= h->cfg.max_keyframes) { h->err = "keyframe slot out of range"; return ELLC_ERR_INVALID; }
        if (h->kf_state[slots[i]] == 0) { h->err = "keyframe slot empty"; return ELLC_ERR_NOT_READY; }
    }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    if (h->uploads_pending) CU_TRY(h, cudaStreamWaitEvent(h->stream, h->up_ev, 0));
    return prepare_keyframes_impl(h, n, slots);
}

// Preparation on the preparation stream: it waits for pending uploads and for the last batch that READ any of these slots, not
// for the batch that is tracking now -- so the pyramids / texels / selection lists of batch k+1 are built while batch k tracks.
int ellc_prepare_async(ellc_handle* h, int32_t n_frames, const int32_t* frame_slots, int32_t n_keyframes, const int32_t* kf_slots) {
    if (!h) return ELLC_ERR_INVALID;
    if (n_frames < 0 || n_keyframes < 0 || (n_frames > 0 && !frame_slots) || (n_keyframes > 0 && !kf_slots) ||
        n_frames > h->cfg.max_frames || n_keyframes > h->cfg.max_keyframes) { h->err = "bad slot lists"; return ELLC_ERR_INVALID; }
    long long reader = 0;
    for (int i = 0; i < n_frames; ++i) {
        const int v = frame_slots[i];
        if (v < 0 || v >= h->cfg.max_frames) { h->err = "frame slot out of range"; return ELLC_ERR_INVALID; }
        if (h->fr_state[v] == 0) { h->err = "frame slot empty"; return ELLC_ERR_NOT_READY; }
        reader = std::max(reader, h->fr_reader[v]);
    }
    for (int i = 0; i < n_keyframes; ++i) {
        const int v = kf_slots[i];
        if (v < 0 || v >= h->cfg.max_keyframes) { h->err = "keyframe slot out of range"; return ELLC_ERR_INVALID; }
        if (h->kf_state[v] == 0) { h->err = "keyframe slot empty"; return ELLC_ERR_NOT_READY; }
        reader = std::max(reader, h->kf_reader[v]);
    }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    if (h->uploads_pending) CU_TRY(h, cudaStreamWaitEvent(h->prep_stream, h->up_ev, 0));   // (the flag stays: other consumers wait too)
    if (h->hyp_pending) CU_TRY(h, cudaStreamWaitEvent(h->prep_stream, h->hyp_ev, 0));       // depth pyramids from hypotheses (main stream)
    if (reader > h->batch_done_seq && reader + 4 > h->batch_seq)                            // (an older ring entry was recycled => finished)
        CU_TRY(h, cudaStreamWaitEvent(h->prep_stream, h->batch_ev[reader & 3], 0));
    int rc = prepare_frames_impl(h, n_frames, frame_slots, true);
    if (rc) return rc;
    rc = prepare_keyframes_impl(h, n_keyframes, kf_slots, true);
    if (rc) return rc;
    CU_TRY(h, cudaEventRecord(h->prep_ev, h->prep_stream));
    CU_TRY(h, cudaStreamWaitEvent(h->stream, h->prep_ev, 0));
    return ELLC_OK;
}

int ellc_synchronize(ellc_handle* h) {
    if (!h) return ELLC_ERR_INVALID;
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    return sync_all_streams(h);
}

int ellc_fence(ellc_handle* h) {
    if (!h) return ELLC_ERR_INVALID;
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    return main_waits_batches(h);
}

int ellc_track_batch_async(ellc_handle* h, int32_t n, const ellc_pair* pairs, const ellc_result** device_results) {
    if (!h) return ELLC_ERR_INVALID;
    if (n < 0 || (n > 0 && !pairs)) { h->err = "bad pair list"; return ELLC_ERR_INVALID; }
    int rc = track_launch(h, n, pairs, false);
    if (rc) return rc;
    if (device_results) *device_results = h->d_results;
    return ELLC_OK;
}

int ellc_results_download(ellc_handle* h, const ellc_result* device_results, int32_t n, ellc_result* results) {
    if (!h) return ELLC_ERR_INVALID;
    if (n < 0 || (n > 0 && (!device_results || !results))) { h->err = "bad download arguments"; return ELLC_ERR_INVALID; }
    if (n == 0) return ELLC_OK;
    int which = -1;
    for (int r = 0; r < 4; ++r) if (device_results == h->d_results4[r]) which = r;
    if (which < 0) { h->err = "pointer was not returned by ellc_track_batch_async (or its buffer has been recycled)"; return ELLC_ERR_INVALID; }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    const long long seq = h->res_seq[which];               // the batch that filled this buffer last
    if (seq < 1) { h->err = "no batch has used this buffer yet"; return ELLC_ERR_NOT_READY; }
    if (n > h->ring_cap[which]) { h->err = "more records requested than the batch held"; return ELLC_ERR_INVALID; }
    CU_TRY(h, cudaStreamWaitEvent(h->d2h_stream, h->batch_ev[seq & 3], 0));
    CU_TRY(h, cudaMemcpyAsync(results, device_results, (size_t)n * sizeof(ellc_result), cudaMemcpyDeviceToHost, h->d2h_stream));
    CU_TRY(h, cudaStreamSynchronize(h->d2h_stream));
    note_done(h, seq);
    h->res_taken[which] = true;
    return ELLC_OK;
}

int ellc_track_batch(ellc_handle* h, int32_t n, const ellc_pair* pairs, ellc_result* results, ellc_iter_trace* trace) {
    if (!h) return ELLC_ERR_INVALID;
    if (n < 0 || (n > 0 && (!pairs || !results))) { h->err = "bad pair list / null results"; return ELLC_ERR_INVALID; }
    if (n == 0) return ELLC_OK;
    int rc = track_launch(h, n, pairs, trace != nullptr);
    if (rc) return rc;
    cudaStream_t ts = h->tstream[h->batch_seq & 1];
    CU_TRY(h, cudaMemcpyAsync(results, h->d_results, (size_t)n * sizeof(ellc_result), cudaMemcpyDeviceToHost, ts));
    if (trace) CU_TRY(h, cudaMemcpyAsync(trace, h->d_trace, (size_t)n * kLevels * ELLC_MAX_TRACE_ITERS * sizeof(ellc_iter_trace),
                                         cudaMemcpyDeviceToHost, ts));
    CU_TRY(h, cudaStreamSynchronize(ts));
    note_done(h, h->batch_seq);
    h->res_taken[h->batch_seq & 3] = true;
    return ELLC_OK;
}

}  // extern "C"

// The loop-closure part of ellc_track_sequence_lc, validated by its caller; null for ellc_track_sequence_steps.
struct SeqLc {
    int n_kf;
    const ellc_lc_keyframe* kfs;
    ellc_lc_ring_params rp;
    const ellc_lc_ring_entry* ring_in;
    int32_t* n_pairs; ellc_pair* pairs; ellc_lc_stats* stats; int32_t* query_of_pair; ellc_result* lc_results;
    ellc_lc_ring_entry* ring_out;
    std::vector<int> list_off;                             // start of every keyframe's frame list; last entry: total length
    std::vector<int> n_frames;                             // its length (ELLC_PAIR_SAVE_WEIGHTS steps naming the keyframe)
    std::vector<int> ret_kf, ret_fr;                       // kf / frame slots of the retired keyframes, in push order
};

// One batch (sequence number, events, slot read-marks) of `waves` tracking launches on one tracking stream.  The call's own device
// buffer holds, carved by n: the steps and the wave order (sorted position -> step; staged together in one copy), the pair records
// the chain kernel writes, the result records and the world poses (indexed by step, i.e. in input order).  The async result ring
// is not touched.  With lc, the loop-closure inputs are staged in the same copy and the keyframe / ring phase runs on the same
// stream after the last wave: frame lists, weights, loop-closure records, histograms, pushes, walk and pack; then one wait for the
// number of pairs, and their tracking.
static int track_sequence_impl(ellc_handle* h, int32_t n, const ellc_seq_step* steps, ellc_result* results, float* world_poses, SeqLc* lc) {
    // wave of a step: one after the later of its dependencies (a step whose world poses are both given by value: wave 0)
    std::vector<int> wave(n);
    int n_waves = 0;
    bool save_weights = false, const_weight = false;
    std::vector<ellc_pair> pairs(n);
    for (int i = 0; i < n; ++i) {
        const ellc_seq_step& s = steps[i];
        if (s.prev_step < -1 || s.prev_step >= i || s.kf_step < -1 || s.kf_step >= i) {
            h->err = "step " + std::to_string(i) + " depends on a step that does not precede it (-1 <= prev_step, kf_step < i)";
            return ELLC_ERR_INVALID;
        }
        wave[i] = 1 + std::max(s.prev_step < 0 ? -1 : wave[s.prev_step], s.kf_step < 0 ? -1 : wave[s.kf_step]);
        n_waves = std::max(n_waves, wave[i] + 1);
        pairs[i].kf_slot = s.kf_slot; pairs[i].frame_slot = s.frame_slot; pairs[i].flags = s.flags;
        save_weights |= (s.flags & ELLC_PAIR_SAVE_WEIGHTS) != 0;
        const_weight |= (s.flags & ELLC_PAIR_CONST_WEIGHT) != 0;
    }
    int rc = validate_pairs(h, n, pairs.data());
    if (rc) return rc;
    // Schedule: by wave, and inside a wave as track_launch orders a batch (forward pairs first, then frame-major, keyframe-minor).
    // Wave w is [start[2w], start[2w + 2]), its forward pairs [start[2w], start[2w + 1]).
    auto key = [&](int i) { return 2 * wave[i] + ((steps[i].flags & ELLC_PAIR_CONST_WEIGHT) ? 1 : 0); };
    std::vector<int> start(2 * n_waves + 1, 0), order(n);
    for (int i = 0; i < n; ++i) { order[i] = i; ++start[key(i) + 1]; }
    for (int k = 0; k < 2 * n_waves; ++k) start[k + 1] += start[k];
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
        if (key(a) != key(b)) return key(a) < key(b);
        if (steps[a].frame_slot != steps[b].frame_slot) return steps[a].frame_slot < steps[b].frame_slot;
        return steps[a].kf_slot < steps[b].kf_slot;
    });
    const int n_kf = lc ? lc->n_kf : 0, n_ret = lc ? (int)lc->ret_kf.size() : 0;
    const int ring_len = lc ? lc->rp.ring_len : 0, n_ring_e = lc ? lc->rp.n_rings * lc->rp.ring_len : 0;
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    rc = flush_dirty(h);
    if (rc) return rc;
    if (save_weights || const_weight || n_kf > 0) {
        rc = ensure_lc_pools(h);
        if (rc) return rc;
    }
    if (n_ret > 0 && !h->fr_hist) CU_TRY(h, cudaMalloc(&h->fr_hist, (size_t)h->cfg.max_frames * 256 * sizeof(float)));
    long long seq = 0;
    rc = batch_begin(h, &seq);
    if (rc) return rc;
    auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
    // loop-closure inputs, staged behind the order: keyframes, ring_in, prior counts [k][level], list offsets, retired kf / frame slots
    const size_t l_kfs = 0, l_ring = up(l_kfs + (size_t)n_kf * sizeof(ellc_lc_keyframe)), l_prior = up(l_ring + (size_t)n_ring_e * sizeof(ellc_lc_ring_entry)),
                 l_off = up(l_prior + (size_t)n_kf * kLevels * sizeof(int)), l_rkf = up(l_off + (size_t)n_kf * sizeof(int)),
                 l_rfr = up(l_rkf + (size_t)n_ret * sizeof(int)), lc_in = lc ? l_rfr + (size_t)n_ret * sizeof(int) : 0;
    const size_t o_order = up((size_t)n * sizeof(ellc_seq_step)), o_lcin = up(o_order + (size_t)n * sizeof(int)), o_pairs = up(o_lcin + lc_in),
                 o_res = up(o_pairs + (size_t)n * sizeof(ellc_pair)), o_world = up(o_res + (size_t)n * sizeof(ellc_result)),
                 seq_end = o_world + (size_t)n * 6 * sizeof(float);
    // loop-closure outputs and scratch: frame lists, their lengths, pushes, queries, per-query segments, the packed list, its records,
    // the rings after the call
    const size_t cap = (size_t)n_kf * ring_len, n_lists = lc ? (size_t)lc->list_off[n_kf] : 0;
    const size_t o_lists = up(seq_end), o_cnt = up(o_lists + n_lists * sizeof(int)), o_push = up(o_cnt + (size_t)n_kf * sizeof(int)),
                 o_q = up(o_push + (size_t)n_kf * sizeof(ellc_lc_ring_entry)), o_segp = up(o_q + (size_t)n_kf * sizeof(ellc_lc_query)),
                 o_segs = up(o_segp + cap * sizeof(ellc_pair)), o_segc = up(o_segs + cap * sizeof(ellc_lc_stats)),
                 o_lp = up(o_segc + (size_t)n_kf * sizeof(int)), o_ls = up(o_lp + cap * sizeof(ellc_pair)), o_lq = up(o_ls + cap * sizeof(ellc_lc_stats)),
                 o_tot = up(o_lq + cap * sizeof(int)), o_lres = up(o_tot + sizeof(int)), o_rout = up(o_lres + cap * sizeof(ellc_result)),
                 total = lc ? o_rout + (size_t)n_ring_e * sizeof(ellc_lc_ring_entry) : seq_end;
    if (total > h->seq_bytes) {                            // (the previous call has completed: it is synchronous)
        cudaFree(h->d_seq); h->d_seq = nullptr; h->seq_bytes = 0;
        CU_TRY(h, cudaMalloc(&h->d_seq, total));
        h->seq_bytes = total;
    }
    char* const d = h->d_seq;
    const ellc_seq_step* d_steps = reinterpret_cast<const ellc_seq_step*>(d);
    const int* d_order = reinterpret_cast<const int*>(d + o_order);
    ellc_pair* d_pairs = reinterpret_cast<ellc_pair*>(d + o_pairs);
    ellc_result* d_res = reinterpret_cast<ellc_result*>(d + o_res);
    float* d_world = reinterpret_cast<float*>(d + o_world);
    rc = batch_order(h, seq, !h->overlap_batches || save_weights || const_weight || lc != nullptr);
    if (rc) return rc;
    cudaStream_t ts = h->tstream[seq & 1];
    int n_lc = 0;
    auto enqueue = [&]() -> int {
        std::vector<char> stage(o_lcin + lc_in);
        std::memcpy(stage.data(), steps, (size_t)n * sizeof(ellc_seq_step));
        std::memcpy(stage.data() + o_order, order.data(), (size_t)n * sizeof(int));
        if (lc) {
            char* L = stage.data() + o_lcin;
            std::memcpy(L + l_kfs, lc->kfs, (size_t)n_kf * sizeof(ellc_lc_keyframe));
            if (n_ring_e) std::memcpy(L + l_ring, lc->ring_in, (size_t)n_ring_e * sizeof(ellc_lc_ring_entry));
            int* prior = reinterpret_cast<int*>(L + l_prior);
            for (int k = 0; k < n_kf; ++k)
                for (int l = 0; l < kLevels; ++l) prior[kLevels * k + l] = h->kf_wcount[(size_t)lc->kfs[k].kf_slot * kLevels + l];
            std::memcpy(L + l_off, lc->list_off.data(), (size_t)n_kf * sizeof(int));
            if (n_ret) {
                std::memcpy(L + l_rkf, lc->ret_kf.data(), (size_t)n_ret * sizeof(int));
                std::memcpy(L + l_rfr, lc->ret_fr.data(), (size_t)n_ret * sizeof(int));
            }
        }
        int r = stage_h2d_on(h, ts, h->d_seq, stage.data(), stage.size());
        if (r) return r;
        CU_TRY(h, cudaEventRecord(h->ev0r[seq & 3], ts));
        TrackParams p;
        fill_params(h, p);
        p.pairs = d_pairs; p.results = d_res;
        if (n_waves > 0) h->launches += launch_seq_init(ts, d_steps, d_order, d_world, d_pairs, 0, start[2]);      // pair records of wave 0
        for (int w = 0; w < n_waves; ++w) {
            const int b = start[2 * w], m = start[2 * w + 1], e = start[2 * w + 2];
            // each wave is scheduled as ellc_track_batch schedules a batch of its pairs: the same cluster / lockstep choice
            p.order = d_order + b; p.n_pairs = m - b;
            const int cluster = pick_cluster(h, m - b);
            p.pairs_per_cta = pick_pairs_per_cta(h, m - b, cluster);
            int l = launch_track(ts, p, cluster, h->cfg.arithmetic);
            if (l < 0) { h->err = std::string("track kernel launch failed: ") + cudaGetErrorString(cudaGetLastError()); return ELLC_ERR_CUDA; }
            h->launches += l;
            if (e > m) {
                p.order = d_order + m; p.n_pairs = e - m;
                l = launch_track_lc(ts, p, h->cfg.arithmetic);
                if (l < 0) { h->err = std::string("loop-closure track kernel launch failed: ") + cudaGetErrorString(cudaGetLastError()); return ELLC_ERR_CUDA; }
                h->launches += l;
            }
            h->launches += launch_seq_world(ts, d_steps, d_order, d_res, d_world, b, e);
            if (w + 1 < n_waves) h->launches += launch_seq_init(ts, d_steps, d_order, d_world, d_pairs, e, start[2 * w + 4]);
        }
        CU_TRY(h, cudaGetLastError());
        if (!lc) return ELLC_OK;
        // ---- keyframes: weights (all listed), then loop-closure records and histograms of the retired ones
        const char* L = d + o_lcin;
        const ellc_lc_keyframe* d_kfs = reinterpret_cast<const ellc_lc_keyframe*>(L + l_kfs);
        const ellc_lc_ring_entry* d_ring_in = reinterpret_cast<const ellc_lc_ring_entry*>(L + l_ring);
        const int* d_off = reinterpret_cast<const int*>(L + l_off);
        int* d_lists = reinterpret_cast<int*>(d + o_lists);
        int* d_cnt = reinterpret_cast<int*>(d + o_cnt);
        h->launches += launch_seq_kf_lists(ts, d_steps, n, d_kfs, n_kf, d_off, d_lists, d_cnt);
        h->launches += launch_seq_kf_weights(ts, h->kf_weight, h->kf_mask, h->fr_weight, d_kfs, n_kf, d_off, d_lists, d_cnt,
                                             reinterpret_cast<const int*>(L + l_prior), h->geo);
        CU_TRY(h, cudaGetLastError());
        if (n_ret == 0) return ELLC_OK;
        const int* d_rkf = reinterpret_cast<const int*>(L + l_rkf);
        h->launches += launch_lc_prepare(ts, h->kf_geo, h->kf_pix, h->geo.win_off[kLevels], h->kf_count, h->kf_img, h->geo.img_off[kLevels],
                                         h->kf_weight, h->kf_lc, h->kf_lcf, h->kf_lcp, h->kf_lcH, h->K, d_rkf, n_ret, h->geo,
                                         h->cfg.arithmetic == ELLC_ARITH_REFERENCE);
        h->launches += launch_frame_histograms(ts, h->fr_img, h->geo.img_off[kLevels], reinterpret_cast<const int*>(L + l_rfr), n_ret,
                                               h->geo.width * h->geo.height, h->fr_hist);
        // ---- ring: pushes with the chain's world poses, the walk of every query on its ring as of its push, the packed pair list
        ellc_lc_ring_entry* d_push = reinterpret_cast<ellc_lc_ring_entry*>(d + o_push);
        ellc_lc_query* d_q = reinterpret_cast<ellc_lc_query*>(d + o_q);
        h->launches += launch_seq_ring_push(ts, d_kfs, n_kf, d_world, d_ring_in, lc->rp.n_rings, ring_len, d_push, d_q,
                                            reinterpret_cast<ellc_lc_ring_entry*>(d + o_rout));
        const int l = launch_lc_generate_seq(ts, h->fr_hist, d_ring_in, ring_len, d_kfs, n_kf, d_push, d_q, lc->rp.min_match_difference,
                                             lc->rp.match_threshold, lc->rp.max_rel_view_angle, ELLC_PAIR_CONST_WEIGHT,
                                             reinterpret_cast<ellc_pair*>(d + o_segp), reinterpret_cast<ellc_lc_stats*>(d + o_segs),
                                             reinterpret_cast<int*>(d + o_segc), reinterpret_cast<ellc_pair*>(d + o_lp),
                                             reinterpret_cast<ellc_lc_stats*>(d + o_ls), reinterpret_cast<int*>(d + o_lq), reinterpret_cast<int*>(d + o_tot));
        if (l < 0) { h->err = "pair-list kernels: bad launch configuration"; return ELLC_ERR_INVALID; }
        h->launches += l;
        CU_TRY(h, cudaGetLastError());
        // ---- the loop-closure pairs: the one wait of the call, for their number (the grid size), then their tracking
        CU_TRY(h, cudaMemcpyAsync(&n_lc, d + o_tot, sizeof(int), cudaMemcpyDeviceToHost, ts));
        CU_TRY(h, cudaStreamSynchronize(ts));
        if (n_lc > 0) {
            TrackParams q;
            fill_params(h, q);
            q.pairs = reinterpret_cast<const ellc_pair*>(d + o_lp); q.order = nullptr; q.results = reinterpret_cast<ellc_result*>(d + o_lres);
            q.n_pairs = n_lc;
            const int lt = launch_track_lc(ts, q, h->cfg.arithmetic);
            if (lt < 0) { h->err = std::string("loop-closure track kernel launch failed: ") + cudaGetErrorString(cudaGetLastError()); return ELLC_ERR_CUDA; }
            h->launches += lt;
        }
        return ELLC_OK;
    };
    const int enq = enqueue();
    // The batch is closed and its slots read-marked even when a launch failed part way: the waves already queued still read these
    // slots, and later uploads / calls must stay ordered behind them.
    rc = batch_end(h, seq);
    for (int i = 0; i < n; ++i) { h->fr_reader[steps[i].frame_slot] = seq; h->kf_reader[steps[i].kf_slot] = seq; }
    if (lc) {
        for (int k = 0; k < n_kf; ++k) { h->fr_reader[lc->kfs[k].frame_slot] = seq; h->kf_reader[lc->kfs[k].kf_slot] = seq; }
        for (int i = 0; i < n_ring_e; ++i)
            if (lc->ring_in[i].is_valid) { h->fr_reader[lc->ring_in[i].frame_slot] = seq; h->kf_reader[lc->ring_in[i].kf_slot] = seq; }
        // the weights were written (as ellc_accumulate_weights / _finalise_weights / ellc_prepare_keyframes_lc leave them)
        for (int k = 0; k < n_kf; ++k) {
            const int ks = lc->kfs[k].kf_slot;
            for (int l = 0; l < kLevels; ++l) h->kf_wcount[(size_t)ks * kLevels + l] += lc->n_frames[k];
            if (lc->n_frames[k] > 0 || lc->kfs[k].retire_before >= 0) h->kf_lc_ready[ks] = 0;
        }
        if (!enq) {
            for (int ks : lc->ret_kf) h->kf_lc_ready[ks] = 1;
            for (int fs : lc->ret_fr) h->fr_hist_ready[fs] = 1;
        }
    }
    if (enq) return enq;
    if (rc) return rc;
    CU_TRY(h, cudaMemcpyAsync(results, d_res, (size_t)n * sizeof(ellc_result), cudaMemcpyDeviceToHost, ts));
    CU_TRY(h, cudaMemcpyAsync(world_poses, d_world, (size_t)n * 6 * sizeof(float), cudaMemcpyDeviceToHost, ts));
    if (lc) {
        *lc->n_pairs = n_lc;
        if (n_lc > 0) {
            if (lc->pairs) CU_TRY(h, cudaMemcpyAsync(lc->pairs, d + o_lp, (size_t)n_lc * sizeof(ellc_pair), cudaMemcpyDeviceToHost, ts));
            if (lc->stats) CU_TRY(h, cudaMemcpyAsync(lc->stats, d + o_ls, (size_t)n_lc * sizeof(ellc_lc_stats), cudaMemcpyDeviceToHost, ts));
            if (lc->query_of_pair) CU_TRY(h, cudaMemcpyAsync(lc->query_of_pair, d + o_lq, (size_t)n_lc * sizeof(int), cudaMemcpyDeviceToHost, ts));
            if (lc->lc_results) CU_TRY(h, cudaMemcpyAsync(lc->lc_results, d + o_lres, (size_t)n_lc * sizeof(ellc_result), cudaMemcpyDeviceToHost, ts));
        }
        if (n_ring_e) {
            if (n_ret > 0) CU_TRY(h, cudaMemcpyAsync(lc->ring_out, d + o_rout, (size_t)n_ring_e * sizeof(ellc_lc_ring_entry), cudaMemcpyDeviceToHost, ts));
            else std::memmove(lc->ring_out, lc->ring_in, (size_t)n_ring_e * sizeof(ellc_lc_ring_entry));
        }
    }
    CU_TRY(h, cudaStreamSynchronize(ts));
    note_done(h, seq);
    return ELLC_OK;
}

extern "C" {

int ellc_track_sequence_steps(ellc_handle* h, int32_t n, const ellc_seq_step* steps, ellc_result* results, float* world_poses) {
    if (!h) return ELLC_ERR_INVALID;
    if (n < 0 || (n > 0 && (!steps || !results || !world_poses))) { h->err = "bad step list / null outputs"; return ELLC_ERR_INVALID; }
    if (n == 0) return ELLC_OK;
    return track_sequence_impl(h, n, steps, results, world_poses, nullptr);
}

int ellc_track_sequence_lc(ellc_handle* h, int32_t n, const ellc_seq_step* steps, int32_t n_kf, const ellc_lc_keyframe* kfs,
                           const ellc_lc_ring_params* ring_params, const ellc_lc_ring_entry* ring_in,
                           ellc_result* results, float* world_poses, int32_t* n_lc_pairs, ellc_pair* lc_pairs, ellc_lc_stats* lc_stats,
                           int32_t* lc_query_of_pair, ellc_result* lc_results, ellc_lc_ring_entry* ring_out) {
    if (!h) return ELLC_ERR_INVALID;
    if (n < 0 || n_kf < 0 || (n > 0 && (!steps || !results || !world_poses)) || (n_kf > 0 && !kfs) || !ring_params || !n_lc_pairs) {
        h->err = "bad step / keyframe lists or null outputs";
        return ELLC_ERR_INVALID;
    }
    *n_lc_pairs = 0;
    const ellc_lc_ring_params& rp = *ring_params;
    if (rp.n_rings < 0 || (rp.n_rings > 0 && (rp.ring_len < 1 || rp.ring_len > 64 || !ring_in || !ring_out))) {
        h->err = "bad ring parameters (1 <= ring_len <= 64, ring_in / ring_out of n_rings x ring_len entries)";
        return ELLC_ERR_INVALID;
    }
    SeqLc lc;
    lc.n_kf = n_kf; lc.kfs = kfs; lc.rp = rp; lc.ring_in = ring_in;
    lc.n_pairs = n_lc_pairs; lc.pairs = lc_pairs; lc.stats = lc_stats; lc.query_of_pair = lc_query_of_pair; lc.lc_results = lc_results;
    lc.ring_out = ring_out;
    if (rp.n_rings == 0) lc.rp.ring_len = 0;
    // keyframes: slots, world dependency, retirement, ring fields
    std::vector<int> kf_index(h->cfg.max_keyframes, -1);
    for (int k = 0; k < n_kf; ++k) {
        const ellc_lc_keyframe& kf = kfs[k];
        const std::string at = "keyframe entry " + std::to_string(k) + ": ";
        if (kf.kf_slot < 0 || kf.kf_slot >= h->cfg.max_keyframes || kf.frame_slot < 0 || kf.frame_slot >= h->cfg.max_frames) {
            h->err = at + "slot out of range"; return ELLC_ERR_INVALID;
        }
        if (kf_index[kf.kf_slot] >= 0) { h->err = at + "keyframe slot listed twice"; return ELLC_ERR_INVALID; }
        kf_index[kf.kf_slot] = k;
        if (h->kf_state[kf.kf_slot] == 0 || h->fr_state[kf.frame_slot] == 0) { h->err = at + "slot never uploaded"; return ELLC_ERR_NOT_READY; }
        if (kf.world_step < -1 || kf.world_step >= n) { h->err = at + "world_step out of range (-1 <= world_step < n)"; return ELLC_ERR_INVALID; }
        if (kf.retire_before < -1 || kf.retire_before > n) { h->err = at + "retire_before out of range (-1 .. n)"; return ELLC_ERR_INVALID; }
        if (kf.retire_before < 0) continue;
        const int L = rp.ring_len;
        if (kf.ring < 0 || kf.ring >= rp.n_rings || kf.ring_pos < 0 || kf.ring_pos >= L || kf.current_array_id < 0 || kf.current_array_id > L ||
            kf.match_window_beg < 0 || kf.match_window_beg >= L || kf.match_window_end < 0 || kf.match_window_end >= L) {
            h->err = at + "ring / ring position / query window out of range"; return ELLC_ERR_INVALID;
        }
        lc.ret_kf.push_back(kf.kf_slot); lc.ret_fr.push_back(kf.frame_slot);
    }
    // steps: no step may track against a keyframe after its retirement; frame-list lengths
    lc.n_frames.assign(n_kf, 0);
    for (int i = 0; i < n; ++i) {
        const int ks = steps[i].kf_slot;
        if (ks < 0 || ks >= h->cfg.max_keyframes || kf_index[ks] < 0) continue;      // (slots are checked with the steps)
        const ellc_lc_keyframe& kf = kfs[kf_index[ks]];
        if (kf.retire_before >= 0 && i >= kf.retire_before) {
            h->err = "step " + std::to_string(i) + " tracks against keyframe entry " + std::to_string(kf_index[ks]) + ", which is retired before it";
            return ELLC_ERR_INVALID;
        }
        if (steps[i].flags & ELLC_PAIR_SAVE_WEIGHTS) ++lc.n_frames[kf_index[ks]];
    }
    lc.list_off.assign(n_kf + 1, 0);
    for (int k = 0; k < n_kf; ++k) lc.list_off[k + 1] = lc.list_off[k] + lc.n_frames[k];
    // the rings before the call: what ellc_lc_generate_pairs requires of a ring
    for (int i = 0; i < rp.n_rings * lc.rp.ring_len; ++i) {
        if (!ring_in[i].is_valid) continue;
        const int fs = ring_in[i].frame_slot, ks = ring_in[i].kf_slot;
        if (fs < 0 || fs >= h->cfg.max_frames || ks < 0 || ks >= h->cfg.max_keyframes) { h->err = "ring entry references a slot out of range"; return ELLC_ERR_INVALID; }
        if (!h->fr_hist || !h->fr_hist_ready[fs]) { h->err = "ring entry without histogram: call ellc_frame_histograms first"; return ELLC_ERR_NOT_READY; }
        if (h->kf_state[ks] == 0) { h->err = "ring entry references a keyframe slot that was never uploaded"; return ELLC_ERR_NOT_READY; }
        const bool retired_here = kf_index[ks] >= 0 && kfs[kf_index[ks]].retire_before >= 0;
        if (!h->kf_lc_ready[ks] && !retired_here) {
            h->err = "ring entry on a keyframe without finalised weights and loop-closure records (ellc_prepare_keyframes_lc)";
            return ELLC_ERR_NOT_READY;
        }
    }
    if (n == 0 && n_kf == 0) {
        if (rp.n_rings > 0) std::memmove(ring_out, ring_in, (size_t)rp.n_rings * rp.ring_len * sizeof(ellc_lc_ring_entry));
        return ELLC_OK;
    }
    return track_sequence_impl(h, n, steps, results, world_poses, &lc);
}

int ellc_gn_iterate(ellc_handle* h, int32_t kf_slot, int32_t frame_slot, int32_t level, int32_t variant, int32_t update,
                    const float pose[6], ellc_iter_trace* out, float* weight_image, const ellc_display_planes* display) {
    if (!h) return ELLC_ERR_INVALID;
    if (!pose || !out || level < 0 || level >= kLevels || variant < 0 || variant > ELLC_VARIANT_PYRAMID) { h->err = "bad evaluate arguments"; return ELLC_ERR_INVALID; }
    const bool lc = variant == ELLC_VARIANT_CONST_WEIGHT;
    if (lc && (weight_image || display)) { h->err = "the constant-weight variant has no per-iteration weight / display images (src/PixelWisePyramid.cpp:687-913)"; return ELLC_ERR_INVALID; }
    ellc_pair pr;
    pr.kf_slot = kf_slot; pr.frame_slot = frame_slot; pr.flags = lc ? ELLC_PAIR_CONST_WEIGHT : 0;
    for (int i = 0; i < 6; ++i) pr.init_pose[i] = pose[i];
    int rc = validate_pairs(h, 1, &pr);
    if (rc) return rc;
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    rc = flush_dirty(h);
    if (rc) return rc;
    rc = main_waits_batches(h);
    if (rc) return rc;
    if (lc) { rc = ensure_lc_pools(h); if (rc) return rc; }
    if (h->trace_cap < (int64_t)kLevels * ELLC_MAX_TRACE_ITERS) {
        cudaFree(h->d_trace); h->d_trace = nullptr; h->trace_cap = 0;
        CU_TRY(h, cudaMalloc(&h->d_trace, (size_t)kLevels * ELLC_MAX_TRACE_ITERS * sizeof(ellc_iter_trace)));
        h->trace_cap = (int64_t)kLevels * ELLC_MAX_TRACE_ITERS;
    }
    // the evaluation has its own pair / result record (behind the record in d_eval_result): it never touches a batch's buffers
    ellc_pair* d_pair = reinterpret_cast<ellc_pair*>(reinterpret_cast<char*>(h->d_eval_result) + sizeof(ellc_result));
    rc = stage_h2d(h, d_pair, &pr, sizeof(pr));
    if (rc) return rc;
    const int64_t npx = (int64_t)h->geo.cols[level] * h->geo.rows[level];
    const bool want_disp = display && (display->warped_image || display->iteration_residual || display->warped_x || display->warped_y);
    const int64_t need = npx * ((weight_image || want_disp) ? 1 : 0) + npx * (want_disp ? 4 : 0);
    if (need > h->weight_cap) {
        cudaFree(h->d_weight); h->d_weight = nullptr; h->weight_cap = 0;
        CU_TRY(h, cudaMalloc(&h->d_weight, (size_t)h->geo.win_off[1] * 5 * sizeof(float)));
        h->weight_cap = h->geo.win_off[1] * 5;
    }
    float* d_disp = h->d_weight ? h->d_weight + npx : nullptr;
    if (weight_image || want_disp) CU_TRY(h, cudaMemsetAsync(h->d_weight, 0, (size_t)npx * sizeof(float), h->stream));
    if (want_disp) {
        // unselected pixels: display_warpedimg = display_iterationres = 0, savedWarpedPoints = -2 (src/PixelWisePyramid.cpp:207-221)
        CU_TRY(h, cudaMemsetAsync(d_disp, 0, (size_t)npx * 2 * sizeof(float), h->stream));
        h->launches += launch_fill_f32(h->stream, d_disp + 2 * npx, -2.0f, 2 * npx);
    }
    CU_TRY(h, cudaMemsetAsync(h->d_trace, 0, (size_t)kLevels * ELLC_MAX_TRACE_ITERS * sizeof(ellc_iter_trace), h->stream));
    TrackParams p;
    fill_params(h, p);
    p.pairs = d_pair; p.results = h->d_eval_result; p.trace = h->d_trace; p.n_pairs = 1;
    p.level_hi = p.level_lo = level; p.iter_limit = 1; p.no_update = update ? 0 : 1;
    // flavour: the handle's, except that the matrix-form Pyramid.cpp variant and the display planes exist in STRICT (and
    // REFERENCE, which evaluates pixels as STRICT does) only
    int arith = h->cfg.arithmetic;
    if (variant == ELLC_VARIANT_PYRAMID) { arith = ELLC_ARITH_STRICT; p.jacobian_at_warped = 1; }
    if (variant == ELLC_VARIANT_FORWARD && !h->cfg.jacobian_at_warped) p.jacobian_at_warped = 0;
    if (want_disp) { if (arith == ELLC_ARITH_FAST) arith = ELLC_ARITH_STRICT; p.disp_out = d_disp; }
    p.weight_out = (weight_image || want_disp) ? h->d_weight : nullptr;
    const int l = lc ? launch_track_lc(h->stream, p, arith) : launch_track(h->stream, p, pick_cluster(h, 1), arith);
    if (l < 0) { h->err = std::string("track kernel launch failed: ") + cudaGetErrorString(cudaGetLastError()); return ELLC_ERR_CUDA; }
    h->launches += l;
    CU_TRY(h, cudaMemcpyAsync(out, h->d_trace + (int64_t)level * ELLC_MAX_TRACE_ITERS, sizeof(ellc_iter_trace), cudaMemcpyDeviceToHost, h->stream));
    if (weight_image) CU_TRY(h, cudaMemcpyAsync(weight_image, h->d_weight, (size_t)npx * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    if (want_disp) {
        float* dst[4] = {display->warped_image, display->iteration_residual, display->warped_x, display->warped_y};
        for (int k = 0; k < 4; ++k)
            if (dst[k]) CU_TRY(h, cudaMemcpyAsync(dst[k], d_disp + k * npx, (size_t)npx * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    }
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return ELLC_OK;
}

int ellc_gn_evaluate(ellc_handle* h, int32_t kf_slot, int32_t frame_slot, int32_t level, const float pose[6],
                     ellc_iter_trace* out, float* weight_image) {
    if (!h) return ELLC_ERR_INVALID;
    return ellc_gn_iterate(h, kf_slot, frame_slot, level, h->cfg.jacobian_at_warped ? ELLC_VARIANT_PYRAMID : ELLC_VARIANT_FORWARD, 0,
                           pose, out, weight_image, nullptr);
}

int ellc_hessian_inverse(ellc_handle* h, const float H[36], float Hinv[36], int32_t* regular) {
    if (!h) return ELLC_ERR_INVALID;
    if (!H || !Hinv) { h->err = "null argument"; return ELLC_ERR_INVALID; }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    float outv[37];
    int rc = stage_h2d(h, h->d_small, H, 36 * sizeof(float));
    if (rc) return rc;
    h->launches += launch_invert6(h->stream, h->d_small, h->d_small + 64);
    CU_TRY(h, cudaMemcpyAsync(outv, h->d_small + 64, sizeof(outv), cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    for (int i = 0; i < 36; ++i) Hinv[i] = outv[i];
    if (regular) *regular = outv[36] != 0.f ? 1 : 0;
    return ELLC_OK;
}

int ellc_solve_update_rt(ellc_handle* h, const float H[36], const float b[6], const float pose_in[6], float pose_out[6],
                         float delta[6], float* weighted_pose, float rt_out[12]) {
    if (!h) return ELLC_ERR_INVALID;
    if (!H || !b || !pose_in || !pose_out || !delta || !weighted_pose) { h->err = "null argument"; return ELLC_ERR_INVALID; }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    float in[54], outv[27];
    for (int i = 0; i < 36; ++i) in[i] = H[i];
    for (int i = 0; i < 6; ++i) { in[36 + i] = b[i]; in[42 + i] = pose_in[i]; in[48 + i] = h->cfg.weight[i]; }
    int rc = stage_h2d(h, h->d_small, in, sizeof(in));
    if (rc) return rc;
    h->launches += launch_solve_update(h->stream, h->d_small, h->d_small + 64, h->cfg.arithmetic);
    CU_TRY(h, cudaMemcpyAsync(outv, h->d_small + 64, sizeof(outv), cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    for (int i = 0; i < 6; ++i) { pose_out[i] = outv[i]; delta[i] = outv[6 + i]; }
    *weighted_pose = outv[12];
    if (rt_out) for (int i = 0; i < 12; ++i) rt_out[i] = outv[14 + i];
    return ELLC_OK;
}

int ellc_solve_update(ellc_handle* h, const float H[36], const float b[6], const float pose_in[6], float pose_out[6],
                      float delta[6], float* weighted_pose) {
    return ellc_solve_update_rt(h, H, b, pose_in, pose_out, delta, weighted_pose, nullptr);
}

int ellc_level_dims(const ellc_handle* h, int32_t level, int32_t* pyr_w, int32_t* pyr_h, int32_t* cols, int32_t* rows) {
    if (!h || level < 0 || level >= kLevels) return ELLC_ERR_INVALID;
    if (pyr_w) *pyr_w = h->geo.pyr_w[level];
    if (pyr_h) *pyr_h = h->geo.pyr_h[level];
    if (cols) *cols = h->geo.cols[level];
    if (rows) *rows = h->geo.rows[level];
    return ELLC_OK;
}

int ellc_read_frame_level(ellc_handle* h, int32_t slot, int32_t level, uint8_t* image, float* gradx, float* grady) {
    if (!h) return ELLC_ERR_INVALID;
    if (slot < 0 || slot >= h->cfg.max_frames || level < 0 || level >= kLevels) { h->err = "bad slot/level"; return ELLC_ERR_INVALID; }
    if (h->fr_state[slot] == 0) { h->err = "frame slot empty"; return ELLC_ERR_NOT_READY; }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = flush_dirty(h);
    if (rc) return rc;
    { int rcw = main_waits_batches(h); if (rcw) return rcw; }
    const Geometry& g = h->geo;
    if (image) CU_TRY(h, cudaMemcpyAsync(image, h->fr_img + (int64_t)slot * g.img_off[kLevels] + g.img_off[level],
                                         (size_t)g.pyr_w[level] * g.pyr_h[level], cudaMemcpyDeviceToHost, h->stream));
    std::vector<uint32_t> tex;
    const size_t npx = (size_t)g.cols[level] * g.rows[level];
    if (gradx || grady) {
        tex.resize(npx);
        CU_TRY(h, cudaMemcpyAsync(tex.data(), h->fr_tex + (int64_t)slot * (g.win_off[kLevels] + kTexPad) + kTexPad + g.win_off[level], npx * 4,
                                  cudaMemcpyDeviceToHost, h->stream));
    }
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    for (size_t i = 0; i < tex.size(); ++i) {           // unpack only: the differences were taken on the device
        if (gradx) gradx[i] = 0.5f * (float)tex_gx2(tex[i]);
        if (grady) grady[i] = 0.5f * (float)tex_gy2(tex[i]);
    }
    return ELLC_OK;
}

int ellc_read_keyframe_level(ellc_handle* h, int32_t slot, int32_t level, uint8_t* image, uint8_t* mask, int32_t* count) {
    if (!h) return ELLC_ERR_INVALID;
    if (slot < 0 || slot >= h->cfg.max_keyframes || level < 0 || level >= kLevels) { h->err = "bad slot/level"; return ELLC_ERR_INVALID; }
    if (h->kf_state[slot] == 0) { h->err = "keyframe slot empty"; return ELLC_ERR_NOT_READY; }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = flush_dirty(h);
    if (rc) return rc;
    { int rcw = main_waits_batches(h); if (rcw) return rcw; }
    const Geometry& g = h->geo;
    if (image) CU_TRY(h, cudaMemcpyAsync(image, h->kf_img + (int64_t)slot * g.img_off[kLevels] + g.img_off[level],
                                         (size_t)g.pyr_w[level] * g.pyr_h[level], cudaMemcpyDeviceToHost, h->stream));
    if (mask) CU_TRY(h, cudaMemcpyAsync(mask, h->kf_mask + (int64_t)slot * g.win_off[kLevels] + g.win_off[level],
                                        (size_t)g.cols[level] * g.rows[level], cudaMemcpyDeviceToHost, h->stream));
    if (count) CU_TRY(h, cudaMemcpyAsync(count, h->kf_count + slot * kLevels + level, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return ELLC_OK;
}

void ellc_concat_relative(const float a[6], const float b[6], float dest[6]) { concat_relative_f(a, b, dest); }
void ellc_concat_origin(const float a[6], const float b[6], float dest[6]) { concat_origin_f(a, b, dest); }
void ellc_se3_exp(const float pose[6], float T[16]) {
    float Rt[12];
    pose_to_rt_f(pose, Rt);
    for (int i = 0; i < 12; ++i) T[i] = Rt[i];
    T[12] = T[13] = T[14] = 0.f; T[15] = 1.f;
}

// The FAST flavour's closed-form small-angle exponential / logarithm (ellc_lie.cuh), as host code for the CPU tests
void ellc_se3_exp_closed(const float pose[6], float T[16]) {
    float Rt[12];
    se3_exp_small_f(pose, Rt);
    for (int i = 0; i < 12; ++i) T[i] = Rt[i];
    T[12] = T[13] = T[14] = 0.f; T[15] = 1.f;
}
int ellc_se3_log_closed(const float T[16], float pose[6]) {
    float Rt[12];
    for (int i = 0; i < 12; ++i) Rt[i] = T[i];
    return se3_log_small_f(Rt, pose) ? 1 : 0;
}

int64_t ellc_launch_count(const ellc_handle* h) { return h ? h->launches : 0; }
void ellc_reset_launch_count(ellc_handle* h) { if (h) h->launches = 0; }
void* ellc_stream(ellc_handle* h) { return h ? (void*)h->stream : nullptr; }
// ---- keyframe weight pyramid and loop-closure records ---------------------------------------------------------------
static int check_kf(ellc_handle* h, int32_t slot) {
    if (slot < 0 || slot >= h->cfg.max_keyframes) { h->err = "bad keyframe slot"; return ELLC_ERR_INVALID; }
    if (h->kf_state[slot] == 0) { h->err = "keyframe slot empty"; return ELLC_ERR_NOT_READY; }
    return ELLC_OK;
}

int ellc_reset_keyframe_weights(ellc_handle* h, int32_t kf_slot) {
    if (!h) return ELLC_ERR_INVALID;
    if (kf_slot < 0 || kf_slot >= h->cfg.max_keyframes) { h->err = "bad keyframe slot"; return ELLC_ERR_INVALID; }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = ensure_lc_pools(h);
    if (rc) return rc;
    { int rcw = main_waits_batches(h); if (rcw) return rcw; }
    const int64_t win = h->geo.win_off[kLevels];
    CU_TRY(h, cudaMemsetAsync(h->kf_weight + kf_slot * win, 0, (size_t)win * sizeof(float), h->stream));
    for (int l = 0; l < kLevels; ++l) h->kf_wcount[(size_t)kf_slot * kLevels + l] = 0;
    h->kf_lc_ready[kf_slot] = 0;
    return ELLC_OK;
}

int ellc_accumulate_weights(ellc_handle* h, int32_t kf_slot, int32_t n, const int32_t* frame_slots) {
    if (!h) return ELLC_ERR_INVALID;
    int rc = check_kf(h, kf_slot);
    if (rc) return rc;
    if (n < 0 || (n > 0 && !frame_slots) || n > h->slots_cap) { h->err = "bad frame slot list"; return ELLC_ERR_INVALID; }
    for (int i = 0; i < n; ++i)
        if (frame_slots[i] < 0 || frame_slots[i] >= h->cfg.max_frames) { h->err = "frame slot out of range"; return ELLC_ERR_INVALID; }
    if (n == 0) return ELLC_OK;
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    rc = ensure_lc_pools(h);
    if (rc) return rc;
    rc = flush_dirty(h);                                   // the keyframe's mask must be current
    if (rc) return rc;
    { int rcw = main_waits_batches(h); if (rcw) return rcw; }
    rc = stage_h2d(h, h->d_slots, frame_slots, (size_t)n * sizeof(int));
    if (rc) return rc;
    const int64_t win = h->geo.win_off[kLevels];
    h->launches += launch_accumulate_weights(h->stream, h->kf_weight + kf_slot * win, h->kf_mask + kf_slot * win, h->fr_weight, win, h->d_slots, n);
    CU_TRY(h, cudaGetLastError());
    for (int l = 0; l < kLevels; ++l) h->kf_wcount[(size_t)kf_slot * kLevels + l] += n;          // numWeightsAdded[level]++ per frame
    h->kf_lc_ready[kf_slot] = 0;
    return ELLC_OK;
}

int ellc_finalise_weights(ellc_handle* h, int32_t kf_slot) {
    if (!h) return ELLC_ERR_INVALID;
    int rc = check_kf(h, kf_slot);
    if (rc) return rc;
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    rc = ensure_lc_pools(h);
    if (rc) return rc;
    { int rcw = main_waits_batches(h); if (rcw) return rcw; }
    h->launches += launch_finalise_weights(h->stream, h->kf_weight + kf_slot * h->geo.win_off[kLevels], &h->kf_wcount[(size_t)kf_slot * kLevels], h->geo);
    CU_TRY(h, cudaGetLastError());
    h->kf_lc_ready[kf_slot] = 0;
    return ELLC_OK;
}

int ellc_upload_keyframe_weights(ellc_handle* h, int32_t kf_slot, const float* const weight[ELLC_LEVELS], const int32_t counts[ELLC_LEVELS]) {
    if (!h) return ELLC_ERR_INVALID;
    if (kf_slot < 0 || kf_slot >= h->cfg.max_keyframes || !weight) { h->err = "bad keyframe slot / null weights"; return ELLC_ERR_INVALID; }
    for (int l = 0; l < kLevels; ++l) if (!weight[l]) { h->err = "null weight level"; return ELLC_ERR_INVALID; }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = ensure_lc_pools(h);
    if (rc) return rc;
    { int rcw = main_waits_batches(h); if (rcw) return rcw; }
    const int64_t win = h->geo.win_off[kLevels];
    for (int l = 0; l < kLevels; ++l) {
        const size_t bytes = (size_t)(h->geo.win_off[l + 1] - h->geo.win_off[l]) * sizeof(float);
        CU_TRY(h, cudaMemcpyAsync(h->kf_weight + kf_slot * win + h->geo.win_off[l], weight[l], bytes, cudaMemcpyHostToDevice, h->stream));
        h->kf_wcount[(size_t)kf_slot * kLevels + l] = counts ? counts[l] : 0;
    }
    CU_TRY(h, cudaStreamSynchronize(h->stream));           // caller-owned pageable buffers may be released on return
    h->kf_lc_ready[kf_slot] = 0;
    return ELLC_OK;
}

int ellc_read_keyframe_weights(ellc_handle* h, int32_t kf_slot, int32_t level, float* weight, int32_t* count) {
    if (!h) return ELLC_ERR_INVALID;
    if (kf_slot < 0 || kf_slot >= h->cfg.max_keyframes || level < 0 || level >= kLevels) { h->err = "bad slot/level"; return ELLC_ERR_INVALID; }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = ensure_lc_pools(h);
    if (rc) return rc;
    { int rcw = main_waits_batches(h); if (rcw) return rcw; }
    const size_t npx = (size_t)(h->geo.win_off[level + 1] - h->geo.win_off[level]);
    if (weight) CU_TRY(h, cudaMemcpyAsync(weight, h->kf_weight + kf_slot * h->geo.win_off[kLevels] + h->geo.win_off[level], npx * sizeof(float),
                                          cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    if (count) *count = h->kf_wcount[(size_t)kf_slot * kLevels + level];
    return ELLC_OK;
}

int ellc_read_frame_weights(ellc_handle* h, int32_t frame_slot, int32_t level, float* weight) {
    if (!h) return ELLC_ERR_INVALID;
    if (frame_slot < 0 || frame_slot >= h->cfg.max_frames || level < 0 || level >= kLevels || !weight) { h->err = "bad slot/level"; return ELLC_ERR_INVALID; }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = ensure_lc_pools(h);
    if (rc) return rc;
    { int rcw = main_waits_batches(h); if (rcw) return rcw; }
    const size_t npx = (size_t)(h->geo.win_off[level + 1] - h->geo.win_off[level]);
    CU_TRY(h, cudaMemcpyAsync(weight, h->fr_weight + frame_slot * h->geo.win_off[kLevels] + h->geo.win_off[level], npx * sizeof(float),
                              cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return ELLC_OK;
}

int ellc_prepare_keyframes_lc(ellc_handle* h, int32_t n, const int32_t* kf_slots) {
    if (!h) return ELLC_ERR_INVALID;
    if (n < 0 || (n > 0 && !kf_slots) || n > h->slots_cap) { h->err = "bad keyframe slot list"; return ELLC_ERR_INVALID; }
    for (int i = 0; i < n; ++i) { int rc = check_kf(h, kf_slots[i]); if (rc) return rc; }
    if (n == 0) return ELLC_OK;
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = ensure_lc_pools(h);
    if (rc) return rc;
    rc = flush_dirty(h);                                   // selection lists of the current depth
    if (rc) return rc;
    { int rcw = main_waits_batches(h); if (rcw) return rcw; }
    int* d_slots = h->d_slots + h->slots_cap;
    rc = stage_h2d(h, d_slots, kf_slots, (size_t)n * sizeof(int));
    if (rc) return rc;
    h->launches += launch_lc_prepare(h->stream, h->kf_geo, h->kf_pix, h->geo.win_off[kLevels], h->kf_count, h->kf_img, h->geo.img_off[kLevels],
                                     h->kf_weight, h->kf_lc, h->kf_lcf, h->kf_lcp, h->kf_lcH, h->K, d_slots, n, h->geo,
                                     h->cfg.arithmetic == ELLC_ARITH_REFERENCE);
    CU_TRY(h, cudaGetLastError());
    for (int i = 0; i < n; ++i) h->kf_lc_ready[kf_slots[i]] = 1;
    return ELLC_OK;
}

// The pipelined form (see ellc_prepare_async): on the low-priority preparation stream, behind the last batch that read these
// keyframe slots only, so that it overlaps the batch that is tracking now.
int ellc_prepare_keyframes_lc_async(ellc_handle* h, int32_t n, const int32_t* kf_slots) {
    if (!h) return ELLC_ERR_INVALID;
    if (n < 0 || (n > 0 && !kf_slots) || n > h->slots_cap) { h->err = "bad keyframe slot list"; return ELLC_ERR_INVALID; }
    long long reader = 0;
    for (int i = 0; i < n; ++i) {
        int rc = check_kf(h, kf_slots[i]);
        if (rc) return rc;
        if (h->kf_state[kf_slots[i]] != 2) { h->err = "keyframe slot not prepared (ellc_prepare_async / ellc_prepare_keyframes first)"; return ELLC_ERR_NOT_READY; }
        reader = std::max(reader, h->kf_reader[kf_slots[i]]);
    }
    if (n == 0) return ELLC_OK;
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    int rc = ensure_lc_pools(h);
    if (rc) return rc;
    // weights written on the main stream (accumulate / finalise / upload) are ordered in front of the preparation stream
    CU_TRY(h, cudaEventRecord(h->main_ev, h->stream));
    CU_TRY(h, cudaStreamWaitEvent(h->prep_stream, h->main_ev, 0));
    if (reader > h->batch_done_seq && reader + 4 > h->batch_seq)
        CU_TRY(h, cudaStreamWaitEvent(h->prep_stream, h->batch_ev[reader & 3], 0));
    int* d_slots = h->d_slots_p + h->slots_cap;
    rc = stage_h2d_on(h, h->prep_stream, d_slots, kf_slots, (size_t)n * sizeof(int));
    if (rc) return rc;
    h->launches += launch_lc_prepare(h->prep_stream, h->kf_geo, h->kf_pix, h->geo.win_off[kLevels], h->kf_count, h->kf_img, h->geo.img_off[kLevels],
                                     h->kf_weight, h->kf_lc, h->kf_lcf, h->kf_lcp, h->kf_lcH, h->K, d_slots, n, h->geo,
                                     h->cfg.arithmetic == ELLC_ARITH_REFERENCE);
    CU_TRY(h, cudaGetLastError());
    CU_TRY(h, cudaEventRecord(h->prep_ev, h->prep_stream));
    CU_TRY(h, cudaStreamWaitEvent(h->stream, h->prep_ev, 0));
    for (int i = 0; i < n; ++i) h->kf_lc_ready[kf_slots[i]] = 1;
    return ELLC_OK;
}

int ellc_selftest_division(ellc_handle* h, int64_t n, uint64_t seed, int64_t mismatches[2]) {
    if (!h) return ELLC_ERR_INVALID;
    if (n < 0 || !mismatches) { h->err = "bad self-test arguments"; return ELLC_ERR_INVALID; }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    unsigned long long* d = reinterpret_cast<unsigned long long*>(h->d_small);
    CU_TRY(h, cudaMemsetAsync(d, 0, 2 * sizeof(unsigned long long), h->stream));
    h->launches += launch_div_selftest(h->stream, (long long)n, (unsigned long long)seed, d);
    unsigned long long out[2] = {0, 0};
    CU_TRY(h, cudaMemcpyAsync(out, d, sizeof(out), cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    mismatches[0] = (int64_t)out[0]; mismatches[1] = (int64_t)out[1];
    return ELLC_OK;
}
int ellc_selftest_unzero(ellc_handle* h, int64_t n, uint64_t seed, int64_t* mismatches) {
    if (!h) return ELLC_ERR_INVALID;
    if (n < 0 || !mismatches) { h->err = "bad self-test arguments"; return ELLC_ERR_INVALID; }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    unsigned long long* d = reinterpret_cast<unsigned long long*>(h->d_small);
    CU_TRY(h, cudaMemsetAsync(d, 0, sizeof(unsigned long long), h->stream));
    h->launches += launch_unzero_selftest(h->stream, (long long)n, (unsigned long long)seed, d);
    unsigned long long out = 0;
    CU_TRY(h, cudaMemcpyAsync(&out, d, sizeof(out), cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    *mismatches = (int64_t)out;
    return ELLC_OK;
}
void* ellc_stream_of(ellc_handle* h, int32_t which) {
    if (!h) return nullptr;
    return which == 1 ? (void*)h->copy_stream : which == 2 ? (void*)h->d2h_stream : which == 3 ? (void*)h->tstream[0]
         : which == 4 ? (void*)h->tstream[1] : (void*)h->stream;
}
float ellc_last_track_kernel_ms(ellc_handle* h) { return ellc_batch_kernel_ms(h, 0); }

float ellc_batch_kernel_ms(ellc_handle* h, int32_t batches_ago) {
    if (!h || !h->ev_valid || batches_ago < 0 || batches_ago > 3 || h->batch_seq - batches_ago < 1) return -1.f;
    float ms = -1.f;
    const int r = (int)((h->batch_seq - batches_ago) & 3);
    if (cudaEventSynchronize(h->ev1r[r]) != cudaSuccess) return -1.f;
    if (cudaEventElapsedTime(&ms, h->ev0r[r], h->ev1r[r]) != cudaSuccess) return -1.f;
    return ms;
}

float ellc_batch_interval_ms(ellc_handle* h, int32_t batches_ago) {
    if (!h || !h->ev_valid || batches_ago < 0 || batches_ago > 2 || h->batch_seq - batches_ago < 2) return -1.f;
    float ms = -1.f;
    const int r = (int)((h->batch_seq - batches_ago) & 3), q = (int)((h->batch_seq - batches_ago - 1) & 3);
    if (cudaEventSynchronize(h->ev1r[r]) != cudaSuccess) return -1.f;
    if (cudaEventElapsedTime(&ms, h->ev1r[q], h->ev1r[r]) != cudaSuccess) return -1.f;
    return ms;
}

}  // extern "C"

// =====================================================================================================================
// Multi-GPU result exchange
// =====================================================================================================================
static XchgHeader* xchg_header(const ellc_exchange* xc, int d) { return reinterpret_cast<XchgHeader*>(xc->peer_block[d]); }
static ellc_result* xchg_table(const ellc_exchange* xc, int d, int r) {
    return reinterpret_cast<ellc_result*>(reinterpret_cast<char*>(xc->peer_block[d]) + sizeof(XchgHeader)) + (size_t)r * xc->capacity;
}
static void exchange_release(ellc_handle* h) {
    ellc_exchange* xc = h->xc;
    if (!xc) return;
    for (int d = 0; d < xc->world; ++d)
        if (xc->peer_ipc[d] && xc->peer_block[d]) cudaIpcCloseMemHandle(xc->peer_block[d]);
    cudaFree(xc->block);
    cudaFree(xc->d_ctr);
    if (xc->h_poll) cudaFreeHost(xc->h_poll);
    delete xc;
    h->xc = nullptr;
}
// one 8-byte read of a counter in this or a peer GPU's memory, through the download stream
static int xchg_read_counter(ellc_handle* h, const unsigned long long* dev, unsigned long long* out) {
    CU_TRY(h, cudaMemcpyAsync(h->xc->h_poll, dev, sizeof(unsigned long long), cudaMemcpyDefault, h->d2h_stream));
    CU_TRY(h, cudaStreamSynchronize(h->d2h_stream));
    *out = *h->xc->h_poll;
    return ELLC_OK;
}
static int xchg_poll_until(ellc_handle* h, const unsigned long long* dev, unsigned long long want, double timeout_s, const char* what) {
    const auto t0 = std::chrono::steady_clock::now();
    for (int spins = 0;; ++spins) {
        unsigned long long v = 0;
        int rc = xchg_read_counter(h, dev, &v);
        if (rc) return rc;
        if (v >= want) return ELLC_OK;
        if (std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() > timeout_s) {
            h->err = std::string("result exchange timed out waiting for ") + what +
                     " (every rank must call ellc_track_batch_exchange / ellc_exchange_wait for every token, in order)";
            return ELLC_ERR_NOT_READY;
        }
        if (spins > 4) std::this_thread::sleep_for(std::chrono::microseconds(20));
    }
}
static int xchg_finish_attach(ellc_handle* h) {
    ellc_exchange* xc = h->xc;
    std::vector<unsigned long long*> ptrs((size_t)kXchgRing * ELLC_MAX_RANKS, nullptr);
    for (int r = 0; r < kXchgRing; ++r)
        for (int d = 0; d < xc->world; ++d) ptrs[(size_t)r * ELLC_MAX_RANKS + d] = &xchg_header(xc, d)->arrived[r];
    if (!xc->d_ctr) CU_TRY(h, cudaMalloc(&xc->d_ctr, ptrs.size() * sizeof(unsigned long long*)));
    CU_TRY(h, cudaMemcpy(xc->d_ctr, ptrs.data(), ptrs.size() * sizeof(unsigned long long*), cudaMemcpyHostToDevice));
    xc->attached = true;
    return ELLC_OK;
}

extern "C" {

int ellc_exchange_create(ellc_handle* h, int32_t rank, int32_t world, int32_t capacity, uint8_t ipc_handle[ELLC_IPC_HANDLE_BYTES]) {
    if (!h) return ELLC_ERR_INVALID;
    if (world < 1 || world > ELLC_MAX_RANKS || rank < 0 || rank >= world || capacity < 1) { h->err = "bad rank / world / capacity"; return ELLC_ERR_INVALID; }
    if (h->xc) { h->err = "this handle already has an exchange"; return ELLC_ERR_INVALID; }
    static_assert(sizeof(cudaIpcMemHandle_t) == ELLC_IPC_HANDLE_BYTES, "ELLC_IPC_HANDLE_BYTES");
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    ellc_exchange* xc = new (std::nothrow) ellc_exchange();
    if (!xc) { h->err = "out of host memory"; return ELLC_ERR_INVALID; }
    xc->rank = rank; xc->world = world; xc->capacity = capacity;
    h->xc = xc;
    const size_t bytes = sizeof(XchgHeader) + (size_t)kXchgRing * capacity * sizeof(ellc_result);
    cudaError_t e = cudaMalloc(&xc->block, bytes);
    if (e == cudaSuccess) e = cudaMemset(xc->block, 0, bytes);
    if (e == cudaSuccess) e = cudaHostAlloc(reinterpret_cast<void**>(&xc->h_poll), 64, cudaHostAllocDefault);
    if (e != cudaSuccess) { h->err = std::string("exchange allocation: ") + cudaGetErrorString(e); exchange_release(h); return ELLC_ERR_CUDA; }
    xc->peer_block[rank] = xc->block;
    if (ipc_handle) {
        cudaIpcMemHandle_t ih;
        std::memset(&ih, 0, sizeof(ih));
        e = cudaIpcGetMemHandle(&ih, xc->block);
        if (e != cudaSuccess) {                            // same-process attachment (ellc_exchange_attach_local) still works
            (void)cudaGetLastError();
            std::memset(&ih, 0, sizeof(ih));
            h->err = std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e);
        }
        std::memcpy(ipc_handle, &ih, sizeof(ih));
    }
    return ELLC_OK;
}

int ellc_exchange_attach_ipc(ellc_handle* h, const uint8_t* ipc_handles) {
    if (!h) return ELLC_ERR_INVALID;
    if (!h->xc || !ipc_handles) { h->err = "no exchange / null handles"; return ELLC_ERR_INVALID; }
    ellc_exchange* xc = h->xc;
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    for (int d = 0; d < xc->world; ++d) {
        if (d == xc->rank || xc->peer_block[d]) continue;
        cudaIpcMemHandle_t ih;
        std::memcpy(&ih, ipc_handles + (size_t)d * ELLC_IPC_HANDLE_BYTES, sizeof(ih));
        void* ptr = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&ptr, ih, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            h->err = std::string("cudaIpcOpenMemHandle(rank ") + std::to_string(d) + "): " + cudaGetErrorString(e);
            return ELLC_ERR_CUDA;
        }
        xc->peer_block[d] = ptr;
        xc->peer_ipc[d] = true;
    }
    return xchg_finish_attach(h);
}

int ellc_exchange_attach_local(ellc_handle* h, ellc_handle* const* peers) {
    if (!h) return ELLC_ERR_INVALID;
    if (!h->xc || !peers) { h->err = "no exchange / null peer list"; return ELLC_ERR_INVALID; }
    ellc_exchange* xc = h->xc;
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    for (int d = 0; d < xc->world; ++d) {
        if (d == xc->rank) continue;
        ellc_handle* q = peers[d];
        if (!q || !q->xc || q->xc->rank != d || q->xc->world != xc->world || q->xc->capacity != xc->capacity) {
            h->err = "peer handle without a matching exchange (same world size and capacity, rank = its index)"; return ELLC_ERR_INVALID;
        }
        if (q->cfg.device != h->cfg.device) {
            int can = 0;
            CU_TRY(h, cudaDeviceCanAccessPeer(&can, h->cfg.device, q->cfg.device));
            if (!can) { h->err = "no peer access between the two devices"; return ELLC_ERR_CUDA; }
            cudaError_t e = cudaDeviceEnablePeerAccess(q->cfg.device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { h->err = std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e); return ELLC_ERR_CUDA; }
            (void)cudaGetLastError();
        }
        xc->peer_block[d] = q->xc->block;
        xc->peer_ipc[d] = false;
    }
    return xchg_finish_attach(h);
}

int ellc_exchange_destroy(ellc_handle* h) {
    if (!h) return ELLC_ERR_INVALID;
    cudaSetDevice(h->cfg.device);
    for (int i = 0; i < 2; ++i) cudaStreamSynchronize(h->tstream[i]);
    cudaStreamSynchronize(h->d2h_stream);
    exchange_release(h);
    return ELLC_OK;
}

int ellc_track_batch_exchange(ellc_handle* h, int32_t n, const ellc_pair* pairs, const int32_t* global_index, int32_t n_total,
                              int32_t root, int64_t* token) {
    if (!h) return ELLC_ERR_INVALID;
    ellc_exchange* xc = h->xc;
    if (!xc || !xc->attached) { h->err = "no attached exchange: ellc_exchange_create + ellc_exchange_attach_* first"; return ELLC_ERR_NOT_READY; }
    if (n < 0 || (n > 0 && (!pairs || !global_index)) || !token) { h->err = "bad exchange batch arguments"; return ELLC_ERR_INVALID; }
    if (n_total < n || n_total > xc->capacity || root < -1 || root >= xc->world) { h->err = "n_total exceeds the exchange capacity / bad root"; return ELLC_ERR_INVALID; }
    for (int i = 0; i < n; ++i)
        if (global_index[i] < 0 || global_index[i] >= n_total) { h->err = "global pair index out of range"; return ELLC_ERR_INVALID; }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    const long long t = xc->token + 1;
    const int r = (int)(t % kXchgRing);
    XchgLaunch xl;
    xl.global_index = global_index;
    const int d0 = root < 0 ? 0 : root, d1 = root < 0 ? xc->world : root + 1;
    for (int d = d0; d < d1; ++d) {
        // flow control: receiver d has copied out the token that used this table last
        if (t > kXchgRing) {
            int rc = xchg_poll_until(h, &xchg_header(xc, d)->released[0], (unsigned long long)(t - kXchgRing), 20.0, "a receiver to release its table");
            if (rc) return rc;
        }
        xl.dst[xl.n_dst++] = xchg_table(xc, d, r);
    }
    int rc = track_launch(h, n, pairs, false, &xl);
    if (rc) return rc;
    cudaStream_t ts = h->tstream[h->batch_seq & 1];
    h->launches += launch_xchg_signal(ts, xc->d_ctr + (size_t)r * ELLC_MAX_RANKS + d0, d1 - d0, (unsigned long long)n);
    CU_TRY(h, cudaGetLastError());
    if (root < 0 || root == xc->rank) xc->expected[r] += (unsigned long long)n_total;
    xc->tok[r].seq = h->batch_seq; xc->tok[r].n = n; xc->tok[r].n_total = n_total; xc->tok[r].root = root;
    xc->token = t;
    *token = t;
    return ELLC_OK;
}

int ellc_exchange_wait(ellc_handle* h, int64_t token, ellc_result* results) {
    if (!h) return ELLC_ERR_INVALID;
    ellc_exchange* xc = h->xc;
    if (!xc || !xc->attached) { h->err = "no attached exchange"; return ELLC_ERR_NOT_READY; }
    if (token < 1 || token > xc->token || token + kXchgRing <= xc->token) { h->err = "unknown or expired exchange token"; return ELLC_ERR_INVALID; }
    CU_TRY(h, cudaSetDevice(h->cfg.device));
    const int r = (int)(token % kXchgRing);
    const ellc_exchange::Tok tk = xc->tok[r];
    CU_TRY(h, cudaEventSynchronize(h->batch_ev[tk.seq & 3]));                  // this rank's own batch
    note_done(h, tk.seq);
    if (tk.root >= 0 && tk.root != xc->rank) return ELLC_OK;                   // not a receiver of this token
    int rc = xchg_poll_until(h, &xchg_header(xc, xc->rank)->arrived[r], xc->expected[r], 30.0, "the records of all ranks");
    if (rc) return rc;
    if (results) CU_TRY(h, cudaMemcpyAsync(results, xchg_table(xc, xc->rank, r), (size_t)tk.n_total * sizeof(ellc_result), cudaMemcpyDeviceToHost, h->d2h_stream));
    CU_TRY(h, cudaStreamSynchronize(h->d2h_stream));
    xc->consumed = token;
    if (h->batch_seq == tk.seq) {                          // nothing queued behind this batch: the GPU is idle, publish now
        rc = xchg_publish(h, h->d2h_stream);
        if (rc) return rc;
    }
    CU_TRY(h, cudaStreamSynchronize(h->d2h_stream));
    return ELLC_OK;
}

}  // extern "C"
