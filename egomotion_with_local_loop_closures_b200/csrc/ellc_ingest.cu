// ellc_ingest.cu -- camera frame -> level-0 working image (frame::frame(VideoCapture), src/Frame.cpp:34-119, SURVEY 3.1):
// BGR -> gray (CV_BGR2GRAY), lens undistortion (cv::undistort = initUndistortRectifyMap CV_16SC2 + remap INTER_LINEAR,
// BORDER_CONSTANT 0) and resize to the working size (cv::resize INTER_LINEAR), in that order, with OpenCV 3.0.0's integer
// arithmetic (DESIGN.md section 9).  One pass per output pixel: no camera-resolution intermediate image is built.  Only the
// rows / columns the resize taps touch are ever read, so the undistortion map is built and stored at those tap positions only.
#include <algorithm>
#include <cfloat>
#include <climits>
#include <cmath>

#include "ellc_internal.h"

namespace ellc {

// CV_BGR2GRAY of OpenCV 3.0.0 on u8 (imgproc/color.cpp, RGB2Gray<uchar>): yuv_shift = 14
static __device__ __forceinline__ int gray_at(const uint8_t* __restrict__ src, int pitch, int channels, int y, int x) {
    const uint8_t* p = src + (int64_t)y * pitch + (int64_t)x * channels;
    if (channels == 1) return p[0];
    return (p[0] * 1868 + p[1] * 9617 + p[2] * 4899 + 8192) >> 14;
}

// One resize tap (camera row ty, camera column tx) of the undistorted gray image: remapBilinear<FixedPtCast<int, uchar, 15>>
// with the CV_16SC2 map entry of that position; a tap outside the camera image reads 0 (BORDER_CONSTANT, value 0).
static __device__ __forceinline__ int undistorted_tap(const uint8_t* __restrict__ src, int pitch, int channels, int w, int h, uint2 m) {
    const int x0 = (int)(int16_t)(m.x & 0xffffu), y0 = (int)(int16_t)(m.x >> 16);
    const int a = (int)(m.y & 31u), b = (int)((m.y >> 5) & 31u);
    const bool xi0 = x0 >= 0 && x0 < w, xi1 = x0 + 1 >= 0 && x0 + 1 < w;
    const bool yi0 = y0 >= 0 && y0 < h, yi1 = y0 + 1 >= 0 && y0 + 1 < h;
    const int p00 = (yi0 && xi0) ? gray_at(src, pitch, channels, y0, x0) : 0;
    const int p01 = (yi0 && xi1) ? gray_at(src, pitch, channels, y0, x0 + 1) : 0;
    const int p10 = (yi1 && xi0) ? gray_at(src, pitch, channels, y0 + 1, x0) : 0;
    const int p11 = (yi1 && xi1) ? gray_at(src, pitch, channels, y0 + 1, x0 + 1) : 0;
    const int s = p00 * ((32 - a) * (32 - b) * 32) + p01 * (a * (32 - b) * 32) + p10 * ((32 - a) * b * 32) + p11 * (a * b * 32);
    return min(max((s + (1 << 14)) >> 15, 0), 255);
}

// Level-0 image of frame j = jobs[blockIdx.z]: out(dx, dy) = resize of the (undistorted) gray camera image.  cols[dx] / rows[dy]
// are the resize taps (two source indices, two Q11 coefficients); map holds the CV_16SC2 entry of every tap position, row-major
// over (2 * dy + ky, 2 * dx + kx).
__global__ void __launch_bounds__(256) ingest_kernel(const IngestJob* __restrict__ jobs, IngestGeo g, const int4* __restrict__ cols,
                                                     const int4* __restrict__ rows, const uint2* __restrict__ map) {
    const int dx = blockIdx.x * blockDim.x + threadIdx.x, dy = blockIdx.y * blockDim.y + threadIdx.y;
    if (dx >= g.out_w || dy >= g.out_h) return;
    const IngestJob job = jobs[blockIdx.z];
    const int4 c = __ldg(cols + dx), r = __ldg(rows + dy);
    int hsum[2];
#pragma unroll
    for (int ky = 0; ky < 2; ++ky) {
        int t0, t1;
        if (g.undistort) {
            const uint4 m = __ldg(reinterpret_cast<const uint4*>(map + (int64_t)(2 * dy + ky) * (2 * g.out_w) + 2 * dx));
            t0 = undistorted_tap(job.src, g.pitch, g.channels, g.cam_w, g.cam_h, make_uint2(m.x, m.y));
            t1 = undistorted_tap(job.src, g.pitch, g.channels, g.cam_w, g.cam_h, make_uint2(m.z, m.w));
        } else {
            const int ty = ky ? r.y : r.x;
            t0 = gray_at(job.src, g.pitch, g.channels, ty, c.x);
            t1 = gray_at(job.src, g.pitch, g.channels, ty, c.y);
        }
        hsum[ky] = t0 * c.z + t1 * c.w;                                   // HResizeLinear<uchar, int, short>
    }
    // VResizeLinear<uchar, int, short> (VResizeLinearVec_32s8u): ((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2
    const int v = (((r.z * (hsum[0] >> 4)) >> 16) + ((r.w * (hsum[1] >> 4)) >> 16) + 2) >> 2;
    job.dst[(int64_t)dy * g.out_w + dx] = (uint8_t)min(max(v, 0), 255);
}

// initUndistortRectifyMap (OpenCV 3.0.0 imgproc/undistort.cpp) at the tap positions: one thread per tap row runs the row's
// incremental projection (_x += ir[0], ...) over every camera column up to the last tap column, in double without contraction,
// and evaluates the distortion model where a tap column is reached.
__global__ void undistort_map_kernel(IngestGeo g, UndistortParams p, const int4* __restrict__ cols, const int4* __restrict__ rows,
                                     uint2* __restrict__ map) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;                 // tap row 2 * dy + ky
    if (t >= 2 * g.out_h) return;
    const int4 r = rows[t >> 1];
    const double i = (double)((t & 1) ? r.y : r.x);
    const double* ir = p.ir;
    double _x = __dadd_rn(__dmul_rn(i, ir[1]), ir[2]), _y = __dadd_rn(__dmul_rn(i, ir[4]), ir[5]), _w = __dadd_rn(__dmul_rn(i, ir[7]), ir[8]);
    int j = 0;
    for (int k = 0; k < 2 * g.out_w; ++k) {                               // tap columns are non-decreasing in k
        const int4 c = cols[k >> 1];
        const int tj = (k & 1) ? c.y : c.x;
        for (; j < tj; ++j) { _x = __dadd_rn(_x, ir[0]); _y = __dadd_rn(_y, ir[3]); _w = __dadd_rn(_w, ir[6]); }
        const double w = __ddiv_rn(1.0, _w), x = __dmul_rn(_x, w), y = __dmul_rn(_y, w);
        const double x2 = __dmul_rn(x, x), y2 = __dmul_rn(y, y);
        const double r2 = __dadd_rn(x2, y2), _2xy = __dmul_rn(__dmul_rn(2.0, x), y);
        // kr = (1 + ((k3 r2 + k2) r2 + k1) r2) / (1 + ((k6 r2 + k5) r2 + k4) r2) with k4 = k5 = k6 = 0: the divisor is exactly 1
        const double kr = __dadd_rn(1.0, __dmul_rn(__dadd_rn(__dmul_rn(__dadd_rn(__dmul_rn(p.k3, r2), p.k2), r2), p.k1), r2));
        const double u = __dadd_rn(__dmul_rn(p.fx, __dadd_rn(__dadd_rn(__dmul_rn(x, kr), __dmul_rn(p.p1, _2xy)),
                                                            __dmul_rn(p.p2, __dadd_rn(r2, __dmul_rn(2.0, x2))))), p.u0);
        const double v = __dadd_rn(__dmul_rn(p.fy, __dadd_rn(__dadd_rn(__dmul_rn(y, kr), __dmul_rn(p.p1, __dadd_rn(r2, __dmul_rn(2.0, y2)))),
                                                            __dmul_rn(p.p2, _2xy))), p.v0);
        // saturate_cast<int>(u * INTER_TAB_SIZE) = cvRound (round half to even), then (short)(iu >> 5) and the 5-bit fractions
        const double us = fmin(fmax(__dmul_rn(u, 32.0), (double)INT_MIN), (double)INT_MAX);
        const double vs = fmin(fmax(__dmul_rn(v, 32.0), (double)INT_MIN), (double)INT_MAX);
        const int iu = __double2int_rn(us), iv = __double2int_rn(vs);
        const uint32_t xs = (uint16_t)(int16_t)(iu >> 5), ys = (uint16_t)(int16_t)(iv >> 5);
        map[(int64_t)t * (2 * g.out_w) + k] = make_uint2(xs | (ys << 16), (uint32_t)((iv & 31) * 32 + (iu & 31)));
    }
}

// cv::resize INTER_LINEAR coefficient tables along one axis (imgproc/resize.cpp, resize(): the generic branch for an 8U image):
// fx = (float)((d + 0.5) * scale - 0.5), clamped at both borders, ialpha = saturate_cast<short>(cbuf * INTER_RESIZE_COEF_SCALE).
// scale = 1 / (dsize / ssize) as cv::resize derives it from the destination size.  Exactly 2x2 downscaling switches to INTER_AREA
// there, whose (a + b + c + d + 2) >> 2 these tables reproduce (coefficients 1024 / 1024 in both passes).
static void resize_taps(int ssize, int dsize, int4* taps) {
    const double scale = 1.0 / ((double)dsize / ssize);
    for (int d = 0; d < dsize; ++d) {
        float f = (float)((d + 0.5) * scale - 0.5);
        int s = (int)std::floor(f);
        f -= (float)s;
        if (s < 0) { f = 0.f; s = 0; }
        if (s + 1 >= ssize && s >= ssize - 1) { f = 0.f; s = ssize - 1; }
        const float c0 = 1.f - f;
        taps[d] = make_int4(s, std::min(s + 1, ssize - 1), (int)std::lrint(c0 * 2048), (int)std::lrint(f * 2048));
    }
}

int build_resize_taps(int cam_w, int cam_h, int out_w, int out_h, int4* cols, int4* rows) {
    resize_taps(cam_w, out_w, cols);
    resize_taps(cam_h, out_h, rows);
    return 0;
}

// iR = (newK * R).inv() with R = I (Matx33d::inv: Matx_FastInvOp<double, 3>, cofactors times the reciprocal determinant).
// Returns false for a singular matrix.
bool invert3(const double a_[9], double b[9]) {
    auto a = [&](int r, int c) { return a_[3 * r + c]; };
    double d = a(0, 0) * (a(1, 1) * a(2, 2) - a(2, 1) * a(1, 2)) - a(0, 1) * (a(1, 0) * a(2, 2) - a(2, 0) * a(1, 2)) +
               a(0, 2) * (a(1, 0) * a(2, 1) - a(2, 0) * a(1, 1));
    if (d == 0 || !std::isfinite(d)) return false;
    d = 1 / d;
    b[0] = (a(1, 1) * a(2, 2) - a(1, 2) * a(2, 1)) * d;
    b[1] = (a(0, 2) * a(2, 1) - a(0, 1) * a(2, 2)) * d;
    b[2] = (a(0, 1) * a(1, 2) - a(0, 2) * a(1, 1)) * d;
    b[3] = (a(1, 2) * a(2, 0) - a(1, 0) * a(2, 2)) * d;
    b[4] = (a(0, 0) * a(2, 2) - a(0, 2) * a(2, 0)) * d;
    b[5] = (a(0, 2) * a(1, 0) - a(0, 0) * a(1, 2)) * d;
    b[6] = (a(1, 0) * a(2, 1) - a(1, 1) * a(2, 0)) * d;
    b[7] = (a(0, 1) * a(2, 0) - a(0, 0) * a(2, 1)) * d;
    b[8] = (a(0, 0) * a(1, 1) - a(0, 1) * a(1, 0)) * d;
    return true;
}

int launch_undistort_map(cudaStream_t st, const IngestGeo& g, const UndistortParams& p, const int4* d_cols, const int4* d_rows, uint2* d_map) {
    const int n = 2 * g.out_h;
    undistort_map_kernel<<<(n + 63) / 64, 64, 0, st>>>(g, p, d_cols, d_rows, d_map);
    return 1;
}

int launch_ingest(cudaStream_t st, const IngestJob* d_jobs, int n, const IngestGeo& g, const int4* d_cols, const int4* d_rows, const uint2* d_map) {
    if (n <= 0) return 0;
    const dim3 block(32, 8), grid((g.out_w + 31) / 32, (g.out_h + 7) / 8, n);
    ingest_kernel<<<grid, block, 0, st>>>(d_jobs, g, d_cols, d_rows, d_map);
    return 1;
}

}  // namespace ellc

// ---- cv::getOptimalNewCameraMatrix (calib3d, centerPrincipalPoint = false, newImgSize = imgSize) in the form current OpenCV
// runs (cv2 4.x, checked to 1e-9 by tests/test_ingest_oracle.py; DESIGN.md section 9 on the 3.0.0 form) -------------------------
namespace {

// undistortPoints (R = I, no new projection): normalised coordinates, 5 fixed-point iterations
void undistort_points(const double K[9], const double dist[5], double* px, double* py, int n) {
    const double fx = K[0], fy = K[4], ifx = 1. / fx, ify = 1. / fy, cx = K[2], cy = K[5];
    const double k0 = dist[0], k1 = dist[1], k2 = dist[2], k3 = dist[3], k4 = dist[4];
    for (int i = 0; i < n; ++i) {
        double x = px[i], y = py[i];
        const double x0 = x = (x - cx) * ifx;
        const double y0 = y = (y - cy) * ify;
        for (int j = 0; j < 5; ++j) {
            const double r2 = x * x + y * y;
            const double icdist = (1 + ((0. * r2 + 0.) * r2 + 0.) * r2) / (1 + ((k4 * r2 + k1) * r2 + k0) * r2);
            if (icdist < 0) { x = x0; y = y0; break; }
            const double deltaX = 2 * k2 * x * y + k3 * (r2 + 2 * x * x);
            const double deltaY = k2 * (r2 + 2 * y * y) + 2 * k3 * x * y;
            x = (x0 - deltaX) * icdist;
            y = (y0 - deltaY) * icdist;
        }
        px[i] = x; py[i] = y;
    }
}

}  // namespace

extern "C" int ellc_optimal_new_camera_matrix(const double K[9], const double dist[5], int32_t width, int32_t height, double alpha,
                                              double new_K[9]) {
    if (!K || !dist || !new_K || width < 2 || height < 2 || !(K[0] != 0) || !(K[4] != 0)) return ELLC_ERR_INVALID;
    // getUndistortRectangles: a 9 x 9 grid over the pixel centres 0 .. size - 1, undistorted; inscribed and circumscribed rectangles
    const int N = 9;
    double px[N * N], py[N * N];
    for (int y = 0, k = 0; y < N; ++y)
        for (int x = 0; x < N; ++x, ++k) { px[k] = (double)x * (width - 1) / (N - 1); py[k] = (double)y * (height - 1) / (N - 1); }
    undistort_points(K, dist, px, py, N * N);
    double iX0 = -FLT_MAX, iX1 = FLT_MAX, iY0 = -FLT_MAX, iY1 = FLT_MAX;
    double oX0 = FLT_MAX, oX1 = -FLT_MAX, oY0 = FLT_MAX, oY1 = -FLT_MAX;
    for (int y = 0, k = 0; y < N; ++y)
        for (int x = 0; x < N; ++x, ++k) {
            const double X = px[k], Y = py[k];
            oX0 = std::min(oX0, X); oX1 = std::max(oX1, X); oY0 = std::min(oY0, Y); oY1 = std::max(oY1, Y);
            if (x == 0) iX0 = std::max(iX0, X);
            if (x == N - 1) iX1 = std::min(iX1, X);
            if (y == 0) iY0 = std::max(iY0, Y);
            if (y == N - 1) iY1 = std::min(iY1, Y);
        }
    // projections mapping the inner / outer rectangle onto the image, interpolated by alpha
    const double fx0 = (width - 1) / (iX1 - iX0), fy0 = (height - 1) / (iY1 - iY0), cx0 = -fx0 * iX0, cy0 = -fy0 * iY0;
    const double fx1 = (width - 1) / (oX1 - oX0), fy1 = (height - 1) / (oY1 - oY0), cx1 = -fx1 * oX0, cy1 = -fy1 * oY0;
    for (int i = 0; i < 9; ++i) new_K[i] = K[i];
    new_K[0] = fx0 * (1 - alpha) + fx1 * alpha;
    new_K[4] = fy0 * (1 - alpha) + fy1 * alpha;
    new_K[2] = cx0 * (1 - alpha) + cx1 * alpha;
    new_K[5] = cy0 * (1 - alpha) + cy1 * alpha;
    return ELLC_OK;
}
