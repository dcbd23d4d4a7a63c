/*
 * ellc_ingest_oracle.h -- CPU ORACLE for the camera frame -> level-0 working image step (TEST INFRASTRUCTURE ONLY).
 *
 * A dependency-free C++11 restatement, stage by stage on whole images, of what frame::frame(VideoCapture) does before the tracker
 * sees a frame (src/Frame.cpp:34-119, SURVEY 3.1): cv::cvtColor(CV_BGR2GRAY), cv::undistort (= initUndistortRectifyMap CV_16SC2 +
 * remap INTER_LINEAR / BORDER_CONSTANT 0) and cv::resize INTER_LINEAR, plus cv::getOptimalNewCameraMatrix.  Nothing is shared with
 * the product's fused kernel (egomotion_with_local_loop_closures_b200/csrc/ellc_ingest.cu).  Pinned against cv2 by
 * tests/golden/ingest_vectors.npz (tests/test_ingest_oracle.py).
 */
#ifndef ELLC_INGEST_ORACLE_H_
#define ELLC_INGEST_ORACLE_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Camera frame -> level-0 working image, the steps of frame::frame(VideoCapture) (src/Frame.cpp:34-119, SURVEY 3.1) in their
 * OpenCV 3.0.0 form.  Images are u8; `pitch` is the camera image's row stride in bytes; map_xy is [h][w][2] (CV_16SC2), map_frac
 * [h][w] = (v & 31) * 32 + (u & 31). */
void ellc_oracle_bgr2gray(const uint8_t* src, int w, int h, int channels, int pitch, uint8_t* dst);
void ellc_oracle_undistort_map(const double K[9], const double dist[5], const double new_K[9], int w, int h, int16_t* map_xy,
                               uint16_t* map_frac);
void ellc_oracle_remap_u8(const uint8_t* src, int sw, int sh, const int16_t* map_xy, const uint16_t* map_frac, int w, int h, uint8_t* dst);
void ellc_oracle_resize_u8(const uint8_t* src, int sw, int sh, uint8_t* dst, int dw, int dh);
/* gray -> undistort (if set) -> resize to dw x dh */
void ellc_oracle_ingest(const uint8_t* src, int w, int h, int channels, int pitch, int undistort, const double K[9], const double dist[5],
                        const double new_K[9], uint8_t* dst, int dw, int dh);
void ellc_oracle_optimal_new_camera_matrix(const double K[9], const double dist[5], int w, int h, double alpha, double new_K[9]);

#ifdef __cplusplus
}
#endif
#endif /* ELLC_INGEST_ORACLE_H_ */
