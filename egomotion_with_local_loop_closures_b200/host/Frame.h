// Frame.h -- host shim of the reference's `class frame` (src/Frame.h:32-397), restricted to the members the tracking
// path touches.  Same member names and meanings; the work behind constructImagePyramids / calculateGradient /
// calculateNonZeroDepthPts / updationOnPyrChange is done by the B200 library and read back on demand.
#pragma once

#include <string>
#include <vector>

#include "ExternVariable.h"
#include "Mat.h"

using ellc_host::Mat;
using ellc_host::uchar;

class frame {
public:
    frame();
    // replaces frame(VideoCapture): the caller hands over the grayscale, undistorted, resized level-0 image
    // (src/Frame.cpp:45-75 is host I/O and stays with the caller)
    frame(const unsigned char* gray, int width, int height);
    // what frame(VideoCapture) does after decoding: the camera image (BGR as VideoCapture delivers it, or 1 channel; rows
    // contiguous) is converted to gray, undistorted (util::FLAG_DO_UNDISTORTION) and resized to ORIG_COLS x ORIG_ROWS on the GPU
    // (util::configure_camera first)
    frame(const unsigned char* camera_image, int cam_cols, int cam_rows, int channels);
    ~frame();

    int frameId;
    int parentKeyframeId;
    bool isKeyframe;
    int numWeightsAdded[util::MAX_PYRAMID_LEVEL];
    int width, height;

    Mat image;                                            // black and white image
    Mat image_pyramid[util::MAX_PYRAMID_LEVEL];
    Mat depth;
    Mat weight_pyramid[util::MAX_PYRAMID_LEVEL];
    Mat depth_pyramid[util::MAX_PYRAMID_LEVEL];
    Mat gradientx, gradienty;
    Mat mask;                                             // 255: non-zero depth, 0: zero depth
    int currentRows, currentCols;
    int pyrLevel;
    int no_nonZeroDepthPts;

    float poseWrtOrigin[6];                               // wrt KF
    float poseWrtWorld[6];                                // wrt first frame
    float rescaleFactor;

    void constructImagePyramids();                        // src/Frame.cpp:170-182   (GPU: pyrdown_u8_kernel)
    void calculateGradient();                             // src/Frame.cpp:185-285   (GPU: pack_tex_kernel)
    void calculateNonZeroDepthPts();                      // src/Frame.cpp:295-301   (GPU: select_count_kernel)
    void updationOnPyrChange(int level, bool isPrevious = true);   // src/Frame.cpp:316-327
    void initializePose();
    void calculatePoseWrtOrigin(frame* prev_image, float* poseChangeWrtPrevframe, bool frmhomo = false);   // :329-348
    void calculatePoseWrtWorld(frame* prev_image, float* poseChangeWrtPrevframe, bool frmhomo = false);    // :352-372
    void concatenateRelativePose(float* src_1wrt2, float* src_2wrt3, float* dest_1wrt3);                   // :503-530
    void concatenateOriginPose(float* src_1wrt0, float* src_2wrt0, float* dest_1wrt2);                     // :534-562
    void finaliseWeights();                               // src/Frame.cpp:678-695 (+ loop-closure records on the GPU)
    void calculateRandT();                                // src/Frame.cpp:443-471: SE3_Pose = exp(hat(poseWrtWorld)), SE3_R, SE3_T, Sim3_R

    // Bilinear samplers of the CURRENT pyramid level (pyrLevel / currentCols / currentRows) with the reference's per-tap bound tests
    // (floor taps tested on the floored coordinate, ceil taps on the unfloored one; an out-of-bounds tap contributes 0).
    // src/Frame.h:181-279: intensity; returns -1 iff all four taps are out of bounds and checkOutfBound == 1.
    float getInterpolatedElement(float x1, float y1, int checkOutfBound = 0);
    // src/Frame.h:283-394: gradient maps of the current level, s = "gradx" / "grady" (as left by updationOnPyrChange / calculateGradient)
    float getInterpolatedElement(float x1, float y1, const std::string& s);

    // exp(hat(poseWrtWorld)) as plain row-major arrays (the reference holds Eigen::MatrixXf members of the same names)
    float SE3_Pose[16], SE3_R[9], SE3_T[3], Sim3_R[9];

    // residency in the B200 library (not part of the reference surface).  Every host thread that calls the tracker has its own
    // context (an ellc_handle with its own streams and slot pools, src/GlobalOptimize.cpp:241: the loop-closure thread tracks on
    // its own copies of the frames); gpu_ctx names the context the slot numbers below refer to.
    void* gpu_ctx;
    int gpu_frame_slot, gpu_kf_slot;
    unsigned long long gpu_kf_stamp;                      // bumped by depthMap::markDepthUpdated()
    bool gpu_lc_ready;                                    // weights finalised and loop-closure records built
    // where the keyframe's weight_pyramid[] / numWeightsAdded[] are current: 0 = host Mats (PixelWisePyramid::saveWeights through
    // the class surface), 1 = device (GetImagePoseEstimate's saveWeights, accumulated on the GPU)
    int gpu_weights_on_device;
    static int numberOfInstances;
    frame(const frame& other);                            // `new frame(*currentframe)`, src/GlobalOptimize.cpp:181: a copy is not resident anywhere
    frame& operator=(const frame& other);
};
