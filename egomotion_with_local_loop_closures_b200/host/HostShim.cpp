// HostShim.cpp -- C++ host side of the drop-in: the reference's frame / depthMap / PixelWisePyramid / Pyramid /
// GetImagePoseEstimate call surface (same names, argument meaning and post-conditions) implemented on top of the C-ABI
// of include/ellc_gn.h.  The numerical work of the tracking path happens in the CUDA library: every pyramid image, gradient,
// mask, normal equation and pose update is produced there; this file moves buffers and keeps the reference's bookkeeping
// (src/ImageFunc.cpp:92-138 initial pose, :305-307 pose write-back, level-0 post-conditions).  Host arithmetic is limited to
// what the reference's callers do on single pixels or on the keyframe's weight Mats: frame::getInterpolatedElement,
// saveWeights / finaliseWeights on weight_pyramid[] when the caller drives the class surface itself.
//
// Threading (src/GlobalOptimize.cpp:241, :566-568, :862-864): the main thread and the loop-closure thread call the tracker
// concurrently.  Every calling host thread gets its OWN context -- an ellc_handle with its own CUDA streams, device pools and
// slot tables -- so no tracker call ever waits for another thread's call; the only shared state is the registry of contexts
// (locked for a lookup) and, per context, a small lock around its slot tables for the moment a frame object changes hands.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/ellc_gn.h"
#include "DepthPropagation.h"
#include "ExternVariable.h"
#include "Frame.h"
#include "ImageFunc.h"
#include "PixelWisePyramid.h"
#include "Pyramid.h"

// ---- util:: definitions (src/main.cpp:34-60 defaults) ----------------------------------------------------------------
namespace util {
int ORIG_COLS = 480, ORIG_ROWS = 270;                                    // src/ExternVariable.h:50-51 defaults
float ORIG_FX = 1642.405612f / 4, ORIG_FY = 1636.148027f / 4, ORIG_CX = 240.0f, ORIG_CY = 135.0f;
int MAX_ITER[4] = {4, 7, 9, 12};
bool FLAG_DO_PARALLEL_POSE_ESTIMATION = true;
bool FLAG_INITIALIZE_NONZERO_POSE = false;
bool FLAG_DO_CONST_WEIGHT_POSE_ESTIMATION = false;
bool FLAG_DO_LOOP_CLOSURE = false;
bool FLAG_ALTERNATE_GN_RA = false;
bool FLAG_IS_BOOTSTRAP = false;
int BATCH_START_ID = 0;
int BATCH_SIZE = 0;
void configure(int cols, int rows, float fx, float fy, float cx, float cy) {
    ORIG_COLS = cols; ORIG_ROWS = rows; ORIG_FX = fx; ORIG_FY = fy; ORIG_CX = cx; ORIG_CY = cy;
}
bool FLAG_DO_UNDISTORTION = false;
float DIM_FACTOR = 4.0f;
}  // namespace util

namespace {
ellc_camera g_camera;                           // util::configure_camera; applied to every context before its next ingestion
unsigned long long g_camera_stamp = 0;
std::mutex g_camera_mu;
}  // namespace

namespace util {
void configure_camera(int cam_cols, int cam_rows, int channels, const double K[9], const double dist[5], bool undistort,
                      float dim_factor, double alpha) {
    ellc_camera cam;
    std::memset(&cam, 0, sizeof(cam));
    cam.width = cam_cols; cam.height = cam_rows; cam.channels = channels; cam.pitch = cam_cols * channels;
    cam.undistort = undistort ? 1 : 0;
    for (int i = 0; i < 9; ++i) cam.K[i] = K[i];
    for (int i = 0; i < 5; ++i) cam.dist[i] = dist[i];
    if (undistort && ellc_optimal_new_camera_matrix(K, dist, cam_cols, cam_rows, alpha, cam.new_K) != ELLC_OK)
        throw std::runtime_error("configure_camera: invalid camera matrix / size");
    FLAG_DO_UNDISTORTION = undistort;
    DIM_FACTOR = dim_factor;
    const double resize_factor = 1.0 / dim_factor;                      // RESIZE_FACTOR
    ORIG_COLS = (int)std::lrint(cam_cols * resize_factor);                // cv::resize(src, dst, Size(), f, f): round(size * f)
    ORIG_ROWS = (int)std::lrint(cam_rows * resize_factor);
    std::lock_guard<std::mutex> lk(g_camera_mu);
    g_camera = cam;
    ++g_camera_stamp;
}
}  // namespace util

namespace {

const int kFrameSlots = 64, kKfSlots = 48;     // the reference keeps a ring of 43 keyframes (src/ExternVariable.h:161-162)

struct Context {
    ellc_handle* h = nullptr;
    std::mutex table_mu;                        // the slot tables below (a frame may be taken over by another thread's context)
    std::vector<frame*> frame_owner, kf_owner;
    std::vector<unsigned long long> kf_stamp;
    std::vector<char> frame_pinned, kf_pinned;  // slots referenced by the batch being assembled: not evictable
    int next_frame = 0, next_kf = 0;
    int cols = 0, rows = 0;
    unsigned long long camera_stamp = 0;        // g_camera_stamp last passed to ellc_set_camera
};
std::mutex g_registry_mu;
std::vector<Context*> g_contexts;
thread_local Context* t_ctx = nullptr;
thread_local std::string t_err;

[[noreturn]] void fail(const std::string& what) {
    t_err = what + ": " + ((t_ctx && t_ctx->h) ? ellc_last_error_string(t_ctx->h) : ellc_last_error_string(nullptr));
    throw std::runtime_error(t_err);
}

Context* ctx() {
    Context* c = t_ctx;
    if (!c) {
        c = new Context();
        std::lock_guard<std::mutex> lk(g_registry_mu);
        g_contexts.push_back(c);
        t_ctx = c;
    }
    if (c->h && (c->cols != util::ORIG_COLS || c->rows != util::ORIG_ROWS)) {
        std::lock_guard<std::mutex> lk(c->table_mu);
        for (frame* f : c->frame_owner) if (f && f->gpu_ctx == c) f->gpu_frame_slot = -1;
        for (frame* f : c->kf_owner) if (f && f->gpu_ctx == c) { f->gpu_kf_slot = -1; f->gpu_lc_ready = false; }
        ellc_destroy(c->h);
        c->h = nullptr;
    }
    if (!c->h) {
        ellc_config cfg;
        ellc_default_config(&cfg, util::ORIG_COLS, util::ORIG_ROWS);
        cfg.fx = util::ORIG_FX; cfg.fy = util::ORIG_FY; cfg.cx = util::ORIG_CX; cfg.cy = util::ORIG_CY;
        for (int l = 0; l < 4; ++l) cfg.max_iter[l] = util::MAX_ITER[l];
        cfg.huber_d = util::HUBER_D; cfg.camera_pixel_noise_2 = util::CAMERA_PIXEL_NOISE_2;
        for (int i = 0; i < 6; ++i) cfg.weight[i] = util::weight[i];
        cfg.max_frames = kFrameSlots; cfg.max_keyframes = kKfSlots;
        if (ellc_create(&cfg, &c->h) != ELLC_OK) fail("ellc_create");
        std::lock_guard<std::mutex> lk(c->table_mu);
        c->frame_owner.assign(kFrameSlots, nullptr);
        c->kf_owner.assign(kKfSlots, nullptr);
        c->kf_stamp.assign(kKfSlots, 0);
        c->frame_pinned.assign(kFrameSlots, 0);
        c->kf_pinned.assign(kKfSlots, 0);
        c->next_frame = c->next_kf = 0;
        c->cols = util::ORIG_COLS; c->rows = util::ORIG_ROWS;
        c->camera_stamp = 0;
    }
    return c;
}

// f is about to be used in context c: if another thread's context holds it, that context forgets it (its device copy stays
// valid until the slot is reused; f's slot numbers always refer to f->gpu_ctx)
void adopt(frame* f, Context* c) {
    Context* o = static_cast<Context*>(f->gpu_ctx);
    if (o == c) return;
    if (o) {
        std::lock_guard<std::mutex> lk(o->table_mu);
        if (f->gpu_frame_slot >= 0 && f->gpu_frame_slot < (int)o->frame_owner.size() && o->frame_owner[f->gpu_frame_slot] == f) o->frame_owner[f->gpu_frame_slot] = nullptr;
        if (f->gpu_kf_slot >= 0 && f->gpu_kf_slot < (int)o->kf_owner.size() && o->kf_owner[f->gpu_kf_slot] == f) o->kf_owner[f->gpu_kf_slot] = nullptr;
    }
    f->gpu_ctx = c; f->gpu_frame_slot = -1; f->gpu_kf_slot = -1; f->gpu_lc_ready = false;
    // (weights accumulated on the other context's device stay there: the reference's loop-closure thread works on copies made
    // after finaliseWeights, whose host Mats are current)
    f->gpu_weights_on_device = 0;
}

int take_slot(std::vector<frame*>& owner, std::vector<char>& pinned, int& next, bool keyframe) {
    const int n = (int)owner.size();
    for (int tries = 0; tries < n; ++tries) {
        const int s = next;
        next = (next + 1) % n;
        if (pinned[s]) continue;
        if (frame* old = owner[s]) {
            if (keyframe) { old->gpu_kf_slot = -1; old->gpu_lc_ready = false; }
            else old->gpu_frame_slot = -1;
        }
        return s;
    }
    return -1;
}

// util::configure_camera's camera on context c (before an ingestion)
void apply_camera(Context* c) {
    ellc_camera cam;
    unsigned long long stamp;
    {
        std::lock_guard<std::mutex> lk(g_camera_mu);
        cam = g_camera; stamp = g_camera_stamp;
    }
    if (stamp == 0) { t_err = "frame from a camera image: call util::configure_camera first"; throw std::runtime_error(t_err); }
    if (c->camera_stamp == stamp) return;
    if (ellc_set_camera(c->h, &cam) != ELLC_OK) fail("ellc_set_camera");
    c->camera_stamp = stamp;
}

// the frame's slot in this thread's context; a frame that is not resident is uploaded from its image, or -- camera != NULL, at
// construction -- ingested from the camera image
int frame_slot(frame* f, const unsigned char* camera = nullptr) {
    Context* c = ctx();
    adopt(f, c);
    {
        std::lock_guard<std::mutex> lk(c->table_mu);
        if (f->gpu_frame_slot >= 0 && c->frame_owner[f->gpu_frame_slot] == f) return f->gpu_frame_slot;
        const int s = take_slot(c->frame_owner, c->frame_pinned, c->next_frame, false);
        if (s < 0) { t_err = "more distinct frames in one batch than frame slots"; throw std::runtime_error(t_err); }
        c->frame_owner[s] = f; f->gpu_frame_slot = s;
    }
    if (camera) {
        apply_camera(c);
        const int32_t s = f->gpu_frame_slot;
        if (ellc_ingest_frames(c->h, 1, &s, &camera, 0) != ELLC_OK) fail("ellc_ingest_frames");
        if (ellc_read_frame_level(c->h, s, 0, f->image.ptr<uchar>(0), nullptr, nullptr) != ELLC_OK) fail("ellc_read_frame_level");
    } else if (ellc_upload_frame(c->h, f->gpu_frame_slot, f->image.ptr<uchar>(0)) != ELLC_OK) fail("ellc_upload_frame");
    return f->gpu_frame_slot;
}

// the keyframe's slot, allocated (and its device weights reset) if it has none in this context; *fresh tells the caller
int keyframe_slot_alloc(frame* f, bool* fresh) {
    Context* c = ctx();
    adopt(f, c);
    *fresh = false;
    std::lock_guard<std::mutex> lk(c->table_mu);
    if (f->gpu_kf_slot >= 0 && c->kf_owner[f->gpu_kf_slot] == f) return f->gpu_kf_slot;
    const int s = take_slot(c->kf_owner, c->kf_pinned, c->next_kf, true);
    if (s < 0) { t_err = "more distinct keyframes in one batch than keyframe slots"; throw std::runtime_error(t_err); }
    c->kf_owner[s] = f; f->gpu_kf_slot = s; f->gpu_lc_ready = false;
    c->kf_stamp[s] = ~0ull;
    *fresh = true;
    return s;
}

int keyframe_slot(frame* f, depthMap* dm) {
    Context* c = ctx();
    adopt(f, c);
    const bool resident = f->gpu_kf_slot >= 0 && c->kf_owner[f->gpu_kf_slot] == f;
    if (resident && !dm) return f->gpu_kf_slot;                            // mask / count queries reuse what is there
    const unsigned long long stamp = dm ? dm->stamp : 0;
    if (resident && c->kf_stamp[f->gpu_kf_slot] == stamp) return f->gpu_kf_slot;
    bool fresh = false;
    const int s = keyframe_slot_alloc(f, &fresh);
    if (fresh) {
        if (ellc_reset_keyframe_weights(c->h, s) != ELLC_OK) fail("ellc_reset_keyframe_weights");     // a fresh slot holds no weights
        f->gpu_weights_on_device = 0;
    }
    const float* dptr[4]; const float* vptr[4];
    std::vector<float> novar[4];
    for (int l = 0; l < 4; ++l) {
        dptr[l] = f->depth_pyramid[l].ptr<float>(0);                         // Mats: 0 = invalid at every level
        if (dm && dm->depthvararrptr[l]) vptr[l] = dm->depthvararrptr[l];
        else { novar[l].assign((size_t)(c->cols >> l) * (c->rows >> l), -1.0f); vptr[l] = novar[l].data(); }
    }
    if (ellc_upload_keyframe(c->h, s, f->image.ptr<uchar>(0), dptr, vptr) != ELLC_OK) fail("ellc_upload_keyframe");
    if (ellc_synchronize(c->h) != ELLC_OK) fail("ellc_synchronize");             // novar[] dies at scope exit
    c->kf_stamp[s] = stamp;
    if (f->gpu_lc_ready) {                                                   // new depth: the loop-closure records follow it
        const int32_t ks = s;
        if (ellc_prepare_keyframes_lc(c->h, 1, &ks) != ELLC_OK) fail("ellc_prepare_keyframes_lc");
    }
    return s;
}

void level_dims(int level, int& pw, int& ph, int& cols, int& rows) {
    if (ellc_level_dims(ctx()->h, level, &pw, &ph, &cols, &rows) != ELLC_OK) fail("ellc_level_dims");
}

// ---- keyframe weight pyramid: host Mats <-> device --------------------------------------------------------------------------
void weights_to_host(frame* kf) {                                            // before host code touches weight_pyramid[]
    Context* c = ctx();
    if (!kf->gpu_weights_on_device || kf->gpu_ctx != c || kf->gpu_kf_slot < 0) return;
    for (int l = 0; l < util::MAX_PYRAMID_LEVEL; ++l) {
        int32_t cnt = 0;
        if (ellc_read_keyframe_weights(c->h, kf->gpu_kf_slot, l, kf->weight_pyramid[l].ptr<float>(0), &cnt) != ELLC_OK) fail("ellc_read_keyframe_weights");
        kf->numWeightsAdded[l] = cnt;
    }
    kf->gpu_weights_on_device = 0;
}
void weights_to_device(frame* kf, int ks) {                                  // before device code reads / accumulates them
    Context* c = ctx();
    if (kf->gpu_weights_on_device) return;
    const float* wp[4]; int32_t cnt[4];
    for (int l = 0; l < util::MAX_PYRAMID_LEVEL; ++l) { wp[l] = kf->weight_pyramid[l].ptr<float>(0); cnt[l] = kf->numWeightsAdded[l]; }
    if (ellc_upload_keyframe_weights(c->h, ks, wp, cnt) != ELLC_OK) fail("ellc_upload_keyframe_weights");
    kf->gpu_weights_on_device = 1;
    kf->gpu_lc_ready = false;
}
// loop-closure records (steepest-descent rows, hessian, hessianInv: the `iter == 0` precomputation of :917-939) for the
// keyframe's current depth and whatever its weight pyramid holds now
void ensure_lc_records(frame* kf, int ks) {
    if (kf->gpu_lc_ready) return;
    weights_to_device(kf, ks);
    const int32_t s = ks;
    if (ellc_prepare_keyframes_lc(ctx()->h, 1, &s) != ELLC_OK) fail("ellc_prepare_keyframes_lc");
    kf->gpu_lc_ready = true;
}

}  // namespace

namespace ellc_host {
void shutdown() {
    std::lock_guard<std::mutex> lk(g_registry_mu);
    for (Context* c : g_contexts) {
        if (c->h) { ellc_destroy(c->h); c->h = nullptr; }
        std::lock_guard<std::mutex> lk2(c->table_mu);
        for (frame* f : c->frame_owner) if (f && f->gpu_ctx == c) { f->gpu_frame_slot = -1; }
        for (frame* f : c->kf_owner) if (f && f->gpu_ctx == c) { f->gpu_kf_slot = -1; f->gpu_lc_ready = false; f->gpu_weights_on_device = 0; }
        std::fill(c->frame_owner.begin(), c->frame_owner.end(), nullptr);
        std::fill(c->kf_owner.begin(), c->kf_owner.end(), nullptr);
    }
}
const char* last_error() { return t_err.c_str(); }
int context_count() {
    std::lock_guard<std::mutex> lk(g_registry_mu);
    int n = 0;
    for (Context* c : g_contexts) n += c->h ? 1 : 0;
    return n;
}
}  // namespace ellc_host

// ---- frame --------------------------------------------------------------------------------------------------------------
int frame::numberOfInstances = 0;
namespace { void finish_construction(frame* f); }

frame::frame() : frameId(0), parentKeyframeId(0), isKeyframe(false), width(0), height(0), currentRows(0), currentCols(0),
                 pyrLevel(0), no_nonZeroDepthPts(0), rescaleFactor(1.0f), gpu_ctx(nullptr), gpu_frame_slot(-1), gpu_kf_slot(-1),
                 gpu_kf_stamp(0), gpu_lc_ready(false), gpu_weights_on_device(0) {
    for (int i = 0; i < 6; ++i) poseWrtOrigin[i] = poseWrtWorld[i] = 0.0f;
    for (int l = 0; l < util::MAX_PYRAMID_LEVEL; ++l) numWeightsAdded[l] = 0;
    for (int i = 0; i < 16; ++i) SE3_Pose[i] = (i % 5 == 0) ? 1.f : 0.f;
    for (int i = 0; i < 9; ++i) SE3_R[i] = Sim3_R[i] = (i % 4 == 0) ? 1.f : 0.f;
    SE3_T[0] = SE3_T[1] = SE3_T[2] = 0.f;
}

frame::frame(const unsigned char* gray, int w, int h) : frame() {
    frameId = ++numberOfInstances;                                           // src/Frame.cpp:37
    width = w; height = h;
    image = Mat(h, w, ellc_host::CV_8UC1);
    std::memcpy(image.ptr<uchar>(0), gray, (size_t)w * h);
    finish_construction(this);
}

// src/Frame.cpp:45-75 on the GPU: the level-0 image is built in the frame's slot and read back into `image`
frame::frame(const unsigned char* camera_image, int cam_cols, int cam_rows, int channels) : frame() {
    frameId = ++numberOfInstances;
    {
        std::lock_guard<std::mutex> lk(g_camera_mu);
        if (g_camera_stamp == 0 || g_camera.width != cam_cols || g_camera.height != cam_rows || g_camera.channels != channels) {
            t_err = "camera image does not match util::configure_camera"; throw std::runtime_error(t_err);
        }
    }
    width = util::ORIG_COLS; height = util::ORIG_ROWS;
    image = Mat(height, width, ellc_host::CV_8UC1);
    frame_slot(this, camera_image);
    finish_construction(this);
}

namespace {
// the rest of frame::frame after the level-0 image exists (src/Frame.cpp:81-117)
void finish_construction(frame* f) {
    const int w = f->width, h = f->height;
    f->pyrLevel = 0; f->currentCols = w; f->currentRows = h;                 // :81-84
    f->constructImagePyramids();                                             // :103
    f->calculateGradient();                                                  // :104
    f->depth = Mat::zeros(h, w, ellc_host::CV_32FC1);                         // :107-117
    for (int l = 0; l < util::MAX_PYRAMID_LEVEL; ++l) {
        f->depth_pyramid[l] = Mat::zeros(h >> l, w >> l, ellc_host::CV_32FC1);
        f->weight_pyramid[l] = Mat::zeros(h >> l, w >> l, ellc_host::CV_32FC1);
    }
}
}  // namespace

// `new frame(*currentframe)` (src/GlobalOptimize.cpp:181): member-wise copy -- cv::Mat members share their pixels, as in the
// reference -- of a frame that is resident nowhere yet; weights accumulated on the device are pulled into the source's Mats
// first when the copy is made by the thread that owns them (the reference's pushToArray runs on the main thread).
frame::frame(const frame& o) { *this = o; }
frame& frame::operator=(const frame& o) {
    if (this == &o) return *this;
    if (o.gpu_weights_on_device && o.gpu_ctx == t_ctx) weights_to_host(const_cast<frame*>(&o));
    frameId = o.frameId; parentKeyframeId = o.parentKeyframeId; isKeyframe = o.isKeyframe;
    width = o.width; height = o.height;
    image = o.image; depth = o.depth; gradientx = o.gradientx; gradienty = o.gradienty; mask = o.mask;
    for (int l = 0; l < util::MAX_PYRAMID_LEVEL; ++l) {
        numWeightsAdded[l] = o.numWeightsAdded[l];
        image_pyramid[l] = o.image_pyramid[l]; weight_pyramid[l] = o.weight_pyramid[l]; depth_pyramid[l] = o.depth_pyramid[l];
    }
    currentRows = o.currentRows; currentCols = o.currentCols; pyrLevel = o.pyrLevel; no_nonZeroDepthPts = o.no_nonZeroDepthPts;
    for (int i = 0; i < 6; ++i) { poseWrtOrigin[i] = o.poseWrtOrigin[i]; poseWrtWorld[i] = o.poseWrtWorld[i]; }
    rescaleFactor = o.rescaleFactor;
    std::memcpy(SE3_Pose, o.SE3_Pose, sizeof(SE3_Pose)); std::memcpy(SE3_R, o.SE3_R, sizeof(SE3_R));
    std::memcpy(SE3_T, o.SE3_T, sizeof(SE3_T)); std::memcpy(Sim3_R, o.Sim3_R, sizeof(Sim3_R));
    gpu_ctx = nullptr; gpu_frame_slot = -1; gpu_kf_slot = -1; gpu_kf_stamp = 0; gpu_lc_ready = false; gpu_weights_on_device = 0;
    return *this;
}

// frame::finaliseWeights, src/Frame.cpp:678-695 (called when the keyframe is retired, src/main.cpp:431-434): average the saved
// weights (cv::Mat / int = multiplication by the float reciprocal, which the device kernel and the host branch both do), then
// build the keyframe's loop-closure records so that later loop-closure pairs on it run the constant-weight tracker.
// weight_pyramid[] is left holding what the reference would hold.
void frame::finaliseWeights() {
    Context* c = ctx();
    const bool resident = gpu_ctx == c && gpu_kf_slot >= 0 && c->kf_owner[gpu_kf_slot] == this;
    if (gpu_weights_on_device && resident) {
        bool any = false;
        for (int l = 0; l < util::MAX_PYRAMID_LEVEL; ++l) any = any || numWeightsAdded[l] > 0;
        if (!any) std::printf("\nWeights cannot be averaged!!! ");
        const int32_t ks = gpu_kf_slot;
        if (ellc_finalise_weights(c->h, ks) != ELLC_OK) fail("ellc_finalise_weights");
        if (ellc_prepare_keyframes_lc(c->h, 1, &ks) != ELLC_OK) fail("ellc_prepare_keyframes_lc");
        for (int l = 0; l < util::MAX_PYRAMID_LEVEL; ++l)
            if (ellc_read_keyframe_weights(c->h, ks, l, weight_pyramid[l].ptr<float>(0), nullptr) != ELLC_OK) fail("ellc_read_keyframe_weights");
        gpu_lc_ready = true;
        return;
    }
    for (int level = util::MAX_PYRAMID_LEVEL - 1; level >= 0; level--) {
        if (numWeightsAdded[level] > 0) {
            const float inv = 1.0f / (float)numWeightsAdded[level];
            float* w = weight_pyramid[level].ptr<float>(0);
            const size_t n = (size_t)weight_pyramid[level].rows * weight_pyramid[level].cols;
            for (size_t i = 0; i < n; ++i) w[i] = w[i] * inv;
        } else {
            std::printf("\nWeights cannot be averaged!!! ");
        }
    }
    gpu_weights_on_device = 0;
    gpu_lc_ready = false;                                                    // rebuilt from the host Mats at the next loop-closure use
}

frame::~frame() {
    Context* c = static_cast<Context*>(gpu_ctx);
    if (!c) return;
    std::lock_guard<std::mutex> lk(c->table_mu);
    if (gpu_frame_slot >= 0 && gpu_frame_slot < (int)c->frame_owner.size() && c->frame_owner[gpu_frame_slot] == this) c->frame_owner[gpu_frame_slot] = nullptr;
    if (gpu_kf_slot >= 0 && gpu_kf_slot < (int)c->kf_owner.size() && c->kf_owner[gpu_kf_slot] == this) c->kf_owner[gpu_kf_slot] = nullptr;
}

void frame::constructImagePyramids() {
    const int s = frame_slot(this);
    for (int l = 0; l < util::MAX_PYRAMID_LEVEL; ++l) {
        int pw, ph, c, r;
        level_dims(l, pw, ph, c, r);
        image_pyramid[l] = Mat(ph, pw, ellc_host::CV_8UC1);
        if (ellc_read_frame_level(ctx()->h, s, l, image_pyramid[l].ptr<uchar>(0), nullptr, nullptr) != ELLC_OK) fail("ellc_read_frame_level");
    }
}

void frame::calculateGradient() {
    const int s = frame_slot(this);
    gradientx = Mat(currentRows, currentCols, ellc_host::CV_32FC1);
    gradienty = Mat(currentRows, currentCols, ellc_host::CV_32FC1);
    if (ellc_read_frame_level(ctx()->h, s, pyrLevel, nullptr, gradientx.ptr<float>(0), gradienty.ptr<float>(0)) != ELLC_OK) fail("ellc_read_frame_level");
}

void frame::calculateNonZeroDepthPts() {
    const int s = keyframe_slot(this, nullptr);
    int pw, ph, c, r;
    level_dims(pyrLevel, pw, ph, c, r);
    mask = Mat(r, c, ellc_host::CV_8UC1);
    int count = 0;
    if (ellc_read_keyframe_level(ctx()->h, s, pyrLevel, nullptr, mask.ptr<uchar>(0), &count) != ELLC_OK) fail("ellc_read_keyframe_level");
    no_nonZeroDepthPts = count;
}

void frame::updationOnPyrChange(int level, bool isPrevious) {
    pyrLevel = level;
    currentRows = height >> level;                                           // height / pow(2, level), src/Frame.cpp:321-322
    currentCols = width >> level;
    if (isPrevious) calculateNonZeroDepthPts();
    calculateGradient();
}

void frame::initializePose() { for (int i = 0; i < 6; ++i) poseWrtOrigin[i] = 0.0f; }

void frame::concatenateRelativePose(float* a, float* b, float* dest) { ellc_concat_relative(a, b, dest); }
void frame::concatenateOriginPose(float* a, float* b, float* dest) { ellc_concat_origin(a, b, dest); }

void frame::calculatePoseWrtOrigin(frame* prev_image, float* d, bool frmhomo) {
    if (!frmhomo) concatenateRelativePose(d, prev_image->poseWrtOrigin, poseWrtOrigin);
    else for (int i = 0; i < 3; ++i) poseWrtOrigin[i] = prev_image->poseWrtOrigin[i] + d[i];
}
void frame::calculatePoseWrtWorld(frame* prev_image, float* d, bool frmhomo) {
    if (!frmhomo) concatenateRelativePose(d, prev_image->poseWrtWorld, poseWrtWorld);
    else for (int i = 0; i < 3; ++i) poseWrtWorld[i] = prev_image->poseWrtWorld[i] + d[i];
}

// src/Frame.cpp:443-471: SE3_Pose = exp(hat(poseWrtWorld)) (Eigen's Pade .exp(): ellc_se3_exp), its blocks, and Sim3_R
void frame::calculateRandT() {
    ellc_se3_exp(poseWrtWorld, SE3_Pose);
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) { SE3_R[i * 3 + j] = SE3_Pose[i * 4 + j]; Sim3_R[i * 3 + j] = rescaleFactor * SE3_Pose[i * 4 + j]; }
        SE3_T[i] = SE3_Pose[i * 4 + 3];
    }
}

// ---- the reference's bilinear samplers (src/Frame.h:181-394) -------------------------------------------------------------
// The four taps are (floor x, floor y), (ceil x, floor y), (floor x, ceil y), (ceil x, ceil y).  Each has its own bound test on
// [0, cols-1] x [0, rows-1], made with the FLOORED coordinate for a floor tap and the UNFLOORED one for a ceil tap; a tap that
// fails contributes 0.  Weights are the fractional parts; the blend is ((1-wy) top + wy bottom) of ((1-wx) left + wx right).
namespace {
template <typename T>
float sample_quirky(const Mat& img, int cols, int rows, float x1, float y1, int* n_out) {
    const float fx = std::floor(x1), fy = std::floor(y1);
    const float wx = x1 - fx, wy = y1 - fy;
    const float max_x = (float)(cols - 1), max_y = (float)(rows - 1);
    int out = 0;
    auto tap = [&](float tx, float ty, bool ceil_x, bool ceil_y) -> float {
        if (tx < 0 || tx > max_x || ty < 0 || ty > max_y) { ++out; return 0.0f; }
        const int r = ceil_y ? (int)std::ceil(ty) : (int)ty;
        const int c = ceil_x ? (int)std::ceil(tx) : (int)tx;
        return (float)img.ptr<T>(r)[c];
    };
    const float p1 = tap(fx, fy, false, false);
    const float p2 = tap(x1, fy, true, false);
    const float top = ((1 - wx) * p1) + (wx * p2);
    const float p3 = tap(fx, y1, false, true);
    const float p4 = tap(x1, y1, true, true);
    const float btm = ((1 - wx) * p3) + (wx * p4);
    *n_out = out;
    return ((1 - wy) * top) + (wy * btm);
}
}  // namespace

float frame::getInterpolatedElement(float x1, float y1, int checkOutfBound) {
    int out = 0;
    const float v = sample_quirky<uchar>(image_pyramid[pyrLevel], currentCols, currentRows, x1, y1, &out);
    return (out == 4 && checkOutfBound == 1) ? -1.0f : v;                    // :267-270
}

float frame::getInterpolatedElement(float x1, float y1, const std::string& s) {
    if (std::isinf(x1) || std::isinf(y1)) std::printf("\nInf Error in Get Interpolated: x1: %f, y1: %f", x1, y1);
    int out = 0;
    if (s == "gradx") return sample_quirky<float>(gradientx, currentCols, currentRows, x1, y1, &out);
    if (s == "grady") return sample_quirky<float>(gradienty, currentCols, currentRows, x1, y1, &out);
    return 0.0f;
}

// ---- depthMap -----------------------------------------------------------------------------------------------------------
depthMap::depthMap() : keyFrame(nullptr), currentFrame(nullptr), stamp(1) {
    hyp_store_.assign((size_t)util::ORIG_COLS * util::ORIG_ROWS, depthhypothesis());
    currentDepthHypothesis = hyp_store_.data();
    for (int l = 0; l < util::MAX_PYRAMID_LEVEL; ++l) {
        const size_t n = (size_t)(util::ORIG_COLS >> l) * (util::ORIG_ROWS >> l);
        depth_store_[l].assign(n, l == 0 ? -1.0f : 0.0f);
        var_store_[l].assign(n, -1.0f);
        deptharrptr[l] = depth_store_[l].data();
        depthvararrptr[l] = var_store_[l].data();
    }
}

void depthMap::updateDepthImage(bool /*fromKeyFrameCreation*/) {
    const int w = util::ORIG_COLS, h = util::ORIG_ROWS;
    const size_t n = (size_t)w * h;
    std::vector<unsigned char> valid(n), vout(n);
    std::vector<float> idep(n), vs(n);
    for (size_t i = 0; i < n; ++i) {
        valid[i] = currentDepthHypothesis[i].isValid ? 1 : 0;
        idep[i] = currentDepthHypothesis[i].invDepthSmoothed;
        vs[i] = currentDepthHypothesis[i].varianceSmoothed;
    }
    Context* c = ctx();
    frame* f = keyFrame;
    bool fresh = false;
    const int s = keyframe_slot_alloc(f, &fresh);                            // same slot policy as keyframe_slot()
    if (fresh) {
        if (ellc_reset_keyframe_weights(c->h, s) != ELLC_OK) fail("ellc_reset_keyframe_weights");
        f->gpu_weights_on_device = 0;
    }
    if (ellc_upload_keyframe_hypotheses(c->h, s, f->image.ptr<uchar>(0), valid.data(), idep.data(), vs.data(), vout.data()) != ELLC_OK)
        fail("ellc_upload_keyframe_hypotheses");
    for (size_t i = 0; i < n; ++i) currentDepthHypothesis[i].isValid = vout[i] != 0;       // :1279-1282
    for (int l = 0; l < util::MAX_PYRAMID_LEVEL; ++l) {
        if (ellc_read_keyframe_depth(c->h, s, l, f->depth_pyramid[l].ptr<float>(0), depthvararrptr[l]) != ELLC_OK) fail("ellc_read_keyframe_depth");
        const size_t nl = (size_t)(w >> l) * (h >> l);
        const float* d = f->depth_pyramid[l].ptr<float>(0);
        for (size_t i = 0; i < nl; ++i) deptharrptr[l][i] = (l == 0 && depthvararrptr[0][i] < 0) ? -1.0f : d[i];   // deptharrpyr0 uses -1
    }
    std::memcpy(f->depth.ptr<float>(0), f->depth_pyramid[0].ptr<float>(0), n * sizeof(float));
    ++stamp;
    c->kf_stamp[s] = stamp;                                                  // the device copy IS the current one: no re-upload
    if (f->gpu_lc_ready) { const int32_t ks = s; if (ellc_prepare_keyframes_lc(c->h, 1, &ks) != ELLC_OK) fail("ellc_prepare_keyframes_lc"); }
}

float depthMap::calculate_no_of_Seeds(bool /*calculate_on_current*/) {
    float count = 0;
    for (int i = 0; i < util::ORIG_COLS * util::ORIG_ROWS; ++i) count += float(currentDepthHypothesis[i].isValid);
    return count / (util::ORIG_COLS * util::ORIG_ROWS) * 100;
}

// ---- PixelWisePyramid ---------------------------------------------------------------------------------------------------
PixelWisePyramid::PixelWisePyramid(frame* prevframe, frame* currentframe, float* /*pose ignored, as the reference*/, depthMap* dm)
    : pyrlevel(prevframe->pyrLevel), nRows(prevframe->currentRows), nCols(prevframe->currentCols), pose(nullptr),
      weightedPose(0.f), prev_frame(prevframe), current_frame(currentframe), currentDepthMap(dm), fill_display(true),
      want_weight_image(false), residualSum(0.f) {
    for (int i = 0; i < 6; ++i) prevPose[i] = 0.f;
    covarianceDiagonalWts[0] = covarianceDiagonalWts[1] = covarianceDiagonalWts[2] = 100.0f;    // :28-34 (unused)
    covarianceDiagonalWts[3] = covarianceDiagonalWts[4] = covarianceDiagonalWts[5] = 0.01f;
    hessian = Mat::zeros(6, 6, ellc_host::CV_32FC1);
    hessianInv = Mat::zeros(6, 6, ellc_host::CV_32FC1);
    sd_param = Mat::zeros(1, 6, ellc_host::CV_32FC1);
    deltapose = Mat::zeros(1, 6, ellc_host::CV_32FC1);
}
PixelWisePyramid::~PixelWisePyramid() {}

void PixelWisePyramid::putPreviousPose(frame* t) { t->concatenateOriginPose(t->poseWrtWorld, prev_frame->poseWrtWorld, prevPose); }

static void copy_trace(const ellc_iter_trace& it, Mat& hessian, Mat& sd_param, Mat& deltapose, float* pose, float* weightedPose, float* residualSum) {
    std::memcpy(hessian.ptr<float>(0), it.H, sizeof(it.H));
    std::memcpy(sd_param.ptr<float>(0), it.b, sizeof(it.b));
    std::memcpy(deltapose.ptr<float>(0), it.delta, sizeof(it.delta));
    for (int i = 0; i < 6; ++i) pose[i] = it.pose_after[i];
    *weightedPose = it.weighted_pose;
    *residualSum = it.res_sum;
}

// calculatePixelWiseParallel, src/PixelWisePyramid.cpp:416-455: per-pixel pass over three row bands, sums, hessian.inv(), updatePose()
void PixelWisePyramid::calculatePixelWiseParallel() {
    Context* c = ctx();
    const int ks = keyframe_slot(prev_frame, currentDepthMap), fs = frame_slot(current_frame);
    ellc_iter_trace it;
    ellc_display_planes planes = {nullptr, nullptr, nullptr, nullptr};
    float* wimg = nullptr;
    if (fill_display || want_weight_image) { display_weightimg = Mat::zeros(nRows, nCols, ellc_host::CV_32FC1); wimg = display_weightimg.ptr<float>(0); }
    if (fill_display) {
        display_warpedimg = Mat::zeros(nRows, nCols, ellc_host::CV_32FC1);
        display_iterationres = Mat::zeros(nRows, nCols, ellc_host::CV_32FC1);
        savedWarpedPointsX = Mat::zeros(nRows, nCols, ellc_host::CV_32FC1);
        savedWarpedPointsY = Mat::zeros(nRows, nCols, ellc_host::CV_32FC1);
        planes.warped_image = display_warpedimg.ptr<float>(0); planes.iteration_residual = display_iterationres.ptr<float>(0);
        planes.warped_x = savedWarpedPointsX.ptr<float>(0); planes.warped_y = savedWarpedPointsY.ptr<float>(0);
    }
    if (ellc_gn_iterate(c->h, ks, fs, pyrlevel, ELLC_VARIANT_FORWARD, 1, pose, &it, wimg, fill_display ? &planes : nullptr) != ELLC_OK) fail("ellc_gn_iterate");
    copy_trace(it, hessian, sd_param, deltapose, pose, &weightedPose, &residualSum);
    int32_t regular = 0;
    if (ellc_hessian_inverse(c->h, hessian.ptr<float>(0), hessianInv.ptr<float>(0), &regular) != ELLC_OK) fail("ellc_hessian_inverse");
    if (fill_display) {
        // the image members that are plain copies under the keyframe's mask (:207-229): template = CURRENT image, 2bewarped =
        // keyframe image, origres = their difference (uchar arithmetic promoted to int, stored as float)
        display_templateimg = Mat::zeros(nRows, nCols, ellc_host::CV_8UC1);
        display_2bewarpedimg = Mat::zeros(nRows, nCols, ellc_host::CV_8UC1);
        display_origres = Mat::zeros(nRows, nCols, ellc_host::CV_32FC1);
        if (prev_frame->pyrLevel != pyrlevel || prev_frame->mask.empty() || prev_frame->mask.rows != nRows) prev_frame->updationOnPyrChange(pyrlevel);
        for (int y = 0; y < nRows; ++y) {
            const uchar* cur = current_frame->image_pyramid[pyrlevel].ptr<uchar>(y);
            const uchar* prv = prev_frame->image_pyramid[pyrlevel].ptr<uchar>(y);
            const uchar* m = prev_frame->mask.ptr<uchar>(y);
            uchar* t = display_templateimg.ptr<uchar>(y); uchar* w2 = display_2bewarpedimg.ptr<uchar>(y);
            float* o = display_origres.ptr<float>(y);
            for (int x = 0; x < nCols; ++x) {
                if (m[x] == 0) continue;
                t[x] = cur[x]; w2[x] = prv[x]; o[x] = (float)((int)cur[x] - (int)prv[x]);
            }
        }
    }
}

// updatePose, :460-491, from the members (for callers that fill hessian / sd_param themselves)
void PixelWisePyramid::updatePose() {
    Context* c = ctx();
    float out[6], d[6], wp = 0.f;
    int32_t regular = 0;
    if (ellc_hessian_inverse(c->h, hessian.ptr<float>(0), hessianInv.ptr<float>(0), &regular) != ELLC_OK) fail("ellc_hessian_inverse");
    if (ellc_solve_update(c->h, hessian.ptr<float>(0), sd_param.ptr<float>(0), pose, out, d, &wp) != ELLC_OK) fail("ellc_solve_update");
    for (int i = 0; i < 6; ++i) { pose[i] = out[i]; deltapose.ptr<float>(0)[i] = d[i]; }
    weightedPose = wp;
}

// calculatePixelWiseParallelInvCompositional, :917-974.  iter == 0 is the reference's precomputation (steepest-descent rows from
// the KEYFRAME's gradients, hessian = (J w) J^T, hessianInv) for the keyframe's current depth and weight pyramid: on the device
// these are the loop-closure records of ellc_prepare_keyframes_lc, rebuilt here whenever the weights changed.
void PixelWisePyramid::calculatePixelWiseParallelInvCompositional(int iter) {
    Context* c = ctx();
    const int ks = keyframe_slot(prev_frame, currentDepthMap), fs = frame_slot(current_frame);
    if (iter == 0) prev_frame->gpu_lc_ready = prev_frame->gpu_lc_ready && prev_frame->gpu_weights_on_device;     // host Mats may have changed
    ensure_lc_records(prev_frame, ks);
    ellc_iter_trace it;
    if (ellc_gn_iterate(c->h, ks, fs, pyrlevel, ELLC_VARIANT_CONST_WEIGHT, 1, pose, &it, nullptr, nullptr) != ELLC_OK) fail("ellc_gn_iterate");
    copy_trace(it, hessian, sd_param, deltapose, pose, &weightedPose, &residualSum);
    if (iter == 0) {
        int32_t regular = 0;
        if (ellc_hessian_inverse(c->h, hessian.ptr<float>(0), hessianInv.ptr<float>(0), &regular) != ELLC_OK) fail("ellc_hessian_inverse");
    }
}

// saveWeights, :500-552.  useAverageWeights == true (the one the reference uses, src/ImageFunc.cpp:285): display_weightimg is
// aligned with the keyframe, add it to prev_frame->weight_pyramid[pyrlevel] and count it.  false ("not used"): scatter the weights
// to the warped positions of the CURRENT frame's weight image.
void PixelWisePyramid::saveWeights(bool useAverageWeights) {
    if (display_weightimg.empty()) { t_err = "saveWeights: no display_weightimg (run calculatePixelWiseParallel with fill_display or want_weight_image)"; throw std::runtime_error(t_err); }
    if (useAverageWeights) {
        weights_to_host(prev_frame);
        float* acc = prev_frame->weight_pyramid[pyrlevel].ptr<float>(0);
        const float* w = display_weightimg.ptr<float>(0);
        for (size_t i = 0; i < (size_t)nRows * nCols; ++i) acc[i] = acc[i] + w[i];
        prev_frame->numWeightsAdded[pyrlevel]++;
        prev_frame->gpu_lc_ready = false;
        return;
    }
    if (savedWarpedPointsX.empty()) { t_err = "saveWeights(false) needs savedWarpedPointsX / Y (fill_display)"; throw std::runtime_error(t_err); }
    for (int y = 0; y < nRows; ++y) {
        const float* wx = savedWarpedPointsX.ptr<float>(y);
        const float* wy = savedWarpedPointsY.ptr<float>(y);
        const float* dw = display_weightimg.ptr<float>(y);
        for (int x = 0; x < nCols; ++x) {
            const int warpedx = int(std::floor(wx[x])), warpedy = int(std::floor(wy[x]));
            if ((warpedx == -1 && warpedy == -1) || (warpedx == -2 && warpedy == -2)) continue;       // -1 oob, -2 zero depth
            current_frame->weight_pyramid[pyrlevel].ptr<float>(warpedy)[warpedx] = dw[x];
        }
    }
}

// ---- Pyramid (matrix form, src/Pyramid.cpp) ---------------------------------------------------------------------------------
Pyramid::Pyramid(frame* prevframe, frame* currentframe, float* pose_, depthMap* dm)
    : level(prevframe->pyrLevel), pose(pose_), lastErr(0.f), error(0.f), pointUsage(0.f), weightedPose(0.f), prev_frame(prevframe),
      current_frame(currentframe), currentDepthMap(dm) {
    for (int i = 0; i < 6; ++i) prevPose[i] = 0.f;
    covarianceDiagonalWts[0] = covarianceDiagonalWts[1] = covarianceDiagonalWts[2] = 100.0f;    // :28-34 (motion prior: unused)
    covarianceDiagonalWts[3] = covarianceDiagonalWts[4] = covarianceDiagonalWts[5] = 0.01f;
    hessian = Mat::zeros(6, 6, ellc_host::CV_32FC1);
    hessianInv = Mat::zeros(6, 6, ellc_host::CV_32FC1);
    sd_param = Mat::zeros(1, 6, ellc_host::CV_32FC1);
    deltapose = Mat::zeros(1, 6, ellc_host::CV_32FC1);
    const int n = prev_frame->no_nonZeroDepthPts;
    weights = Mat::zeros(1, n, ellc_host::CV_32FC1);
    residual = Mat::zeros(1, n, ellc_host::CV_32FC1);
    warpedImage = Mat::zeros(1, n, ellc_host::CV_32FC1);
    warpedPoints = Mat::zeros(2, n, ellc_host::CV_32FC1);
}

void Pyramid::putPreviousPose(frame* t) { t->concatenateOriginPose(t->poseWrtWorld, prev_frame->poseWrtWorld, prevPose); }

// One evaluation at *pose (calculateWarpedPoints .. calResidualAndWeights, plus the sums calculateHessianInv / updatePose take
// over the points): fills hessian, sd_param and the per-point rows; returns sum w r^2 / N (:694).
float Pyramid::evaluate(bool update) {
    Context* c = ctx();
    const int ks = keyframe_slot(prev_frame, currentDepthMap), fs = frame_slot(current_frame);
    const int rows = prev_frame->currentRows, cols = prev_frame->currentCols;
    std::vector<float> wimg((size_t)rows * cols), warped((size_t)rows * cols), res((size_t)rows * cols), px((size_t)rows * cols), py((size_t)rows * cols);
    ellc_display_planes planes = {warped.data(), res.data(), px.data(), py.data()};
    ellc_iter_trace it;
    if (ellc_gn_iterate(c->h, ks, fs, level, ELLC_VARIANT_PYRAMID, update ? 1 : 0, pose, &it, wimg.data(), &planes) != ELLC_OK) fail("ellc_gn_iterate");
    std::memcpy(hessian.ptr<float>(0), it.H, sizeof(it.H));
    std::memcpy(sd_param.ptr<float>(0), it.b, sizeof(it.b));
    if (update) {
        std::memcpy(deltapose.ptr<float>(0), it.delta, sizeof(it.delta));
        for (int i = 0; i < 6; ++i) pose[i] = it.pose_after[i];
        weightedPose = it.weighted_pose;
    }
    // per-point rows in raster order of the selected pixels (the order calculateWorldPoints collects them, :211-273)
    if (prev_frame->mask.empty() || prev_frame->mask.rows != rows || prev_frame->pyrLevel != level) prev_frame->updationOnPyrChange(level);
    const int n = prev_frame->no_nonZeroDepthPts;
    if (weights.cols != n) {
        weights = Mat::zeros(1, n, ellc_host::CV_32FC1); residual = Mat::zeros(1, n, ellc_host::CV_32FC1);
        warpedImage = Mat::zeros(1, n, ellc_host::CV_32FC1); warpedPoints = Mat::zeros(2, n, ellc_host::CV_32FC1);
    }
    int k = 0;
    for (int y = 0; y < rows && k < n; ++y) {
        const uchar* m = prev_frame->mask.ptr<uchar>(y);
        for (int x = 0; x < cols && k < n; ++x) {
            if (m[x] == 0) continue;
            const size_t i = (size_t)y * cols + x;
            weights.ptr<float>(0)[k] = wimg[i]; residual.ptr<float>(0)[k] = res[i]; warpedImage.ptr<float>(0)[k] = warped[i];
            warpedPoints.ptr<float>(0)[k] = px[i]; warpedPoints.ptr<float>(1)[k] = py[i];
            ++k;
        }
    }
    return n > 0 ? it.res_sum / float(n) : 0.0f;
}

float Pyramid::calResidualAndWeights() { return evaluate(false); }

void Pyramid::performPrecomputation() { lastErr = calResidualAndWeights(); }                    // :700-711

void Pyramid::calculateHessianInv() {                                                            // :153-207 (the sum is part of evaluate())
    int32_t regular = 0;
    if (ellc_hessian_inverse(ctx()->h, hessian.ptr<float>(0), hessianInv.ptr<float>(0), &regular) != ELLC_OK) fail("ellc_hessian_inverse");
}

void Pyramid::updatePose() {                                                                     // :528-553
    float out[6], d[6], wp = 0.f;
    if (ellc_solve_update(ctx()->h, hessian.ptr<float>(0), sd_param.ptr<float>(0), pose, out, d, &wp) != ELLC_OK) fail("ellc_solve_update");
    for (int i = 0; i < 6; ++i) { pose[i] = out[i]; deltapose.ptr<float>(0)[i] = d[i]; }
    weightedPose = wp;
}

float Pyramid::performIterationSteps() {                                                         // :714-726
    calculateHessianInv();
    updatePose();
    error = calResidualAndWeights();
    const float temp = lastErr;
    lastErr = error;
    return error / temp;
}

// ---- GetImagePoseEstimate -------------------------------------------------------------------------------------------------
static void initial_relative_pose(frame* prev_frame, frame* tminus1, float* initial_pose_estimate, bool fromLoopClosure, float pose[6]) {
    // src/ImageFunc.cpp:97-138
    for (int i = 0; i < 6; ++i) pose[i] = 0.0f;
    if (!util::FLAG_INITIALIZE_NONZERO_POSE || fromLoopClosure) {
        prev_frame->concatenateOriginPose(tminus1->poseWrtWorld, prev_frame->poseWrtWorld, pose);
    } else {
        prev_frame->concatenateOriginPose(initial_pose_estimate, prev_frame->poseWrtWorld, pose);
        float pose_trans[6];
        prev_frame->concatenateOriginPose(tminus1->poseWrtWorld, prev_frame->poseWrtWorld, pose_trans);
        pose[3] = pose_trans[3]; pose[4] = pose_trans[4]; pose[5] = pose_trans[5];
    }
}

std::vector<float> GetImagePoseEstimate(frame* prev_frame, frame* current_frame, int /*frame_num*/, depthMap* currDepthMap,
                                        frame* tminus1_prev_frame, float* initial_pose_estimate, bool fromLoopClosure, bool /*homo*/) {
    float pose[6];
    initial_relative_pose(prev_frame, tminus1_prev_frame, initial_pose_estimate, fromLoopClosure, pose);
    {
        Context* c = ctx();
        ellc_pair pr;
        pr.kf_slot = keyframe_slot(prev_frame, currDepthMap);
        pr.frame_slot = frame_slot(current_frame);
        // src/ImageFunc.cpp:241-244: loop-closure pairs use the constant-weight inverse-compositional tracker, with whatever the
        // keyframe's weight pyramid holds; :280-288: sequential tracks save their last weights into the keyframe's pyramid
        const bool cw = util::FLAG_DO_CONST_WEIGHT_POSE_ESTIMATION;
        pr.flags = (cw && fromLoopClosure) ? ELLC_PAIR_CONST_WEIGHT : (cw && !fromLoopClosure) ? ELLC_PAIR_SAVE_WEIGHTS : ELLC_PAIR_DEFAULT;
        if (pr.flags == ELLC_PAIR_CONST_WEIGHT) ensure_lc_records(prev_frame, pr.kf_slot);
        if (pr.flags == ELLC_PAIR_SAVE_WEIGHTS) weights_to_device(prev_frame, pr.kf_slot);
        for (int i = 0; i < 6; ++i) pr.init_pose[i] = pose[i];
        ellc_result res;
        if (ellc_track_batch(c->h, 1, &pr, &res, nullptr) != ELLC_OK) fail("ellc_track_batch");
        for (int i = 0; i < 6; ++i) pose[i] = res.pose[i];
        if (pr.flags == ELLC_PAIR_SAVE_WEIGHTS) {                              // saveWeights(true), src/PixelWisePyramid.cpp:546-548
            const int32_t fs = pr.frame_slot;
            if (ellc_accumulate_weights(c->h, pr.kf_slot, 1, &fs) != ELLC_OK) fail("ellc_accumulate_weights");
            for (int l = 0; l < util::MAX_PYRAMID_LEVEL; ++l) prev_frame->numWeightsAdded[l]++;
            prev_frame->gpu_lc_ready = false;
        }
    }
    // post-conditions the depth module relies on (src/ImageFunc.cpp:158-159 end at level 0)
    prev_frame->updationOnPyrChange(0);
    current_frame->updationOnPyrChange(0, false);
    current_frame->calculatePoseWrtOrigin(prev_frame, pose);                 // :305
    current_frame->calculatePoseWrtWorld(prev_frame, pose);                  // :306
    current_frame->calculateRandT();                                         // :307
    return std::vector<float>(pose, pose + 6);                               // :311-313
}

// Batched form.  The slots a sub-batch references are pinned while it is assembled, so that a slot an earlier pair of the same
// sub-batch uses is never recycled for a later one; a list with more distinct frames / keyframes than there are slots is split
// into consecutive sub-batches (results keep the caller's order).
std::vector<float> ellc_host::TrackPairsBatched(const std::vector<frame*>& keyframes, const std::vector<depthMap*>& depthMaps,
                                                const std::vector<frame*>& frames, const std::vector<float>& init_poses) {
    const size_t n = frames.size();
    if (keyframes.size() != n || depthMaps.size() != n || init_poses.size() != n * 6) { t_err = "TrackPairsBatched: list sizes differ"; throw std::runtime_error(t_err); }
    std::vector<float> out(n * 6);
    Context* c = ctx();
    size_t lo = 0;
    while (lo < n) {
        std::vector<frame*> df, dk;                                          // distinct frames / keyframes of this sub-batch
        size_t hi = lo;
        for (; hi < n; ++hi) {
            const bool nf = std::find(df.begin(), df.end(), frames[hi]) == df.end(), nk = std::find(dk.begin(), dk.end(), keyframes[hi]) == dk.end();
            if ((nf && (int)df.size() == kFrameSlots) || (nk && (int)dk.size() == kKfSlots)) break;
            if (nf) df.push_back(frames[hi]);
            if (nk) dk.push_back(keyframes[hi]);
        }
        std::vector<ellc_pair> pairs(hi - lo);
        std::vector<ellc_result> res(hi - lo);
        for (size_t i = lo; i < hi; ++i) {
            ellc_pair& p = pairs[i - lo];
            p.kf_slot = keyframe_slot(keyframes[i], depthMaps[i]);
            p.frame_slot = frame_slot(frames[i]);
            { std::lock_guard<std::mutex> lk(c->table_mu); c->kf_pinned[p.kf_slot] = 1; c->frame_pinned[p.frame_slot] = 1; }
            p.flags = util::FLAG_DO_CONST_WEIGHT_POSE_ESTIMATION ? ELLC_PAIR_CONST_WEIGHT : ELLC_PAIR_DEFAULT;
            if (p.flags == ELLC_PAIR_CONST_WEIGHT) ensure_lc_records(keyframes[i], p.kf_slot);
            for (int k = 0; k < 6; ++k) p.init_pose[k] = init_poses[i * 6 + k];
        }
        const int rc = ellc_track_batch(c->h, (int)pairs.size(), pairs.data(), res.data(), nullptr);
        {
            std::lock_guard<std::mutex> lk(c->table_mu);
            std::fill(c->kf_pinned.begin(), c->kf_pinned.end(), 0);
            std::fill(c->frame_pinned.begin(), c->frame_pinned.end(), 0);
        }
        if (rc != ELLC_OK) fail("ellc_track_batch");
        for (size_t i = lo; i < hi; ++i) for (int k = 0; k < 6; ++k) out[i * 6 + k] = res[i - lo].pose[k];
        lo = hi;
    }
    return out;
}
