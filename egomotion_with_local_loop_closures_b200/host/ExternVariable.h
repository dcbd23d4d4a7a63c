// ExternVariable.h -- configuration surface of the drop-in host shim.
//
// Mirrors the names of the reference's src/ExternVariable.h (namespace util) for everything the tracking path reads
// (:39-62 sizes and intrinsics, :76 weight[], :148-149 noise / Huber, :176-185 flags, :224-232 thread counts and UNZERO)
// and src/main.cpp:34-60 (MAX_ITER and the mutable flags).  The reference fixes the image size at compile time; here
// ORIG_COLS / ORIG_ROWS / ORIG_F* / ORIG_C* are set once at start-up with util::configure() because the B200 library
// takes them at run time (ellc_config).
#pragma once

#include <string>

namespace util {

static const int KEYFRAME_PROPAGATE_INTERVAL = 8;
static const int MAX_PYRAMID_LEVEL = 4;

extern int ORIG_COLS, ORIG_ROWS;                 // level-0 working size
extern float ORIG_FX, ORIG_FY, ORIG_CX, ORIG_CY;
void configure(int cols, int rows, float fx, float fy, float cx, float cy);

// The camera of frame(camera_image, ...) (src/Frame.cpp:34-119): FLAG_DO_UNDISTORTION and DIM_FACTOR (RESIZE_FACTOR = 1 / DIM_FACTOR) of
// src/ExternVariable.h, and the camera matrix / distortion coefficients the reference hands to cv::undistort.  configure_camera sets
// ORIG_COLS / ORIG_ROWS to the camera size times RESIZE_FACTOR (rounded, as cv::resize sizes its output) and computes the
// undistorted camera matrix with getOptimalNewCameraMatrix(K, dist, size, alpha) (ellc_optimal_new_camera_matrix).
extern bool FLAG_DO_UNDISTORTION;
extern float DIM_FACTOR;
void configure_camera(int cam_cols, int cam_rows, int channels, const double K[9], const double dist[5], bool undistort,
                      float dim_factor, double alpha);

static const float weight[] = {100000.0f, 100000.0f, 100000.0f, 10000.0f, 10000.0f, 10000.0f};
static const float CAMERA_PIXEL_NOISE_2 = 4.0f * 4.0f;
static const float HUBER_D = 3.0f;
static const int NUM_POSE_THREADS = 3;           // kept for source compatibility; the GPU path ignores it

extern int MAX_ITER[4];                          // src/main.cpp:34
extern bool FLAG_DO_PARALLEL_POSE_ESTIMATION;    // must stay true: this shim IS that path
extern bool FLAG_INITIALIZE_NONZERO_POSE;
extern bool FLAG_DO_CONST_WEIGHT_POSE_ESTIMATION;
extern bool FLAG_DO_PARALLEL_CONST_WEIGHT_POSE_EST;  // constant-weight tracks sum over two row bands (src/PixelWisePyramid.cpp:945-951)
                                                 // instead of one (:970); read by ELLC_ARITH_REFERENCE only (ellc_config::lc_bands)
// Arithmetic flavour of the GPU tracker (ELLC_ARITH_FAST, ELLC_ARITH_STRICT or ELLC_ARITH_REFERENCE of ellc_gn.h; default FAST).
// ELLC_ARITH_REFERENCE reproduces the reference's tracker bit for bit, so that poses_orig.txt / matchframes*.txt of a run can be
// diffed against a CPU run of the reference.  Read when a thread's context creates its tracker (and again after a change).
extern int GPU_ARITHMETIC;
extern bool FLAG_DO_LOOP_CLOSURE;
extern bool FLAG_ALTERNATE_GN_RA;                // batch alternation with rotation averaging ("LC" mode, src/main.cpp:89-92)
extern bool FLAG_IS_BOOTSTRAP;
extern int BATCH_START_ID;
extern int BATCH_SIZE;

#define UNZERO(val) (val < 0 ? (val > -1e-10 ? -1e-10 : val) : (val < 1e-10 ? 1e-10 : val))

}  // namespace util
