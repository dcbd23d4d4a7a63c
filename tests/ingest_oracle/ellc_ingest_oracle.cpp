// ellc_ingest_oracle.cpp -- see ellc_ingest_oracle.h (test infrastructure only).
#include "ellc_ingest_oracle.h"

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <vector>

/* ==== camera frame -> level-0 working image (frame::frame(VideoCapture), src/Frame.cpp:34-119; SURVEY 3.1) ====================
 * The four stages in their OpenCV 3.0.0 form, each on a whole image as the reference runs them: cvtColor, undistort (=
 * initUndistortRectifyMap + remap), resize.  Nothing is shared with the product's fused kernel. */
extern "C" {

/* cv::cvtColor(CV_BGR2GRAY) on u8, imgproc/color.cpp RGB2Gray<uchar>: yuv_shift = 14, coefficients B 1868, G 9617, R 4899 */
void ellc_oracle_bgr2gray(const uint8_t* src, int w, int h, int channels, int pitch, uint8_t* dst) {
    for (int y = 0; y < h; ++y)
        for (int x = 0; x < w; ++x) {
            const uint8_t* p = src + (size_t)y * pitch + (size_t)x * channels;
            dst[(size_t)y * w + x] = channels == 1 ? p[0] : (uint8_t)((p[0] * 1868 + p[1] * 9617 + p[2] * 4899 + 8192) >> 14);
        }
}

/* cv::initUndistortRectifyMap(K, dist, R = I, new_K, size, CV_16SC2), imgproc/undistort.cpp: iR = (new_K R).inv() (Matx33d,
 * cofactors / determinant), per row the incremental projection _x += ir[0], radial / tangential model, INTER_TAB_SIZE = 32 */
void ellc_oracle_undistort_map(const double K[9], const double dist[5], const double new_K[9], int w, int h, int16_t* map_xy,
                               uint16_t* map_frac) {
    double a[3][3], ir[9];
    for (int i = 0; i < 9; ++i) a[i / 3][i % 3] = new_K[i];
    double d = a[0][0] * (a[1][1] * a[2][2] - a[2][1] * a[1][2]) - a[0][1] * (a[1][0] * a[2][2] - a[2][0] * a[1][2]) +
               a[0][2] * (a[1][0] * a[2][1] - a[2][0] * a[1][1]);
    d = 1 / d;
    ir[0] = (a[1][1] * a[2][2] - a[1][2] * a[2][1]) * d; ir[1] = (a[0][2] * a[2][1] - a[0][1] * a[2][2]) * d;
    ir[2] = (a[0][1] * a[1][2] - a[0][2] * a[1][1]) * d; ir[3] = (a[1][2] * a[2][0] - a[1][0] * a[2][2]) * d;
    ir[4] = (a[0][0] * a[2][2] - a[0][2] * a[2][0]) * d; ir[5] = (a[0][2] * a[1][0] - a[0][0] * a[1][2]) * d;
    ir[6] = (a[1][0] * a[2][1] - a[1][1] * a[2][0]) * d; ir[7] = (a[0][1] * a[2][0] - a[0][0] * a[2][1]) * d;
    ir[8] = (a[0][0] * a[1][1] - a[0][1] * a[1][0]) * d;
    const double u0 = K[2], v0 = K[5], fx = K[0], fy = K[4];
    const double k1 = dist[0], k2 = dist[1], p1 = dist[2], p2 = dist[3], k3 = dist[4], k4 = 0, k5 = 0, k6 = 0;
    for (int i = 0; i < h; ++i) {
        double _x = i * ir[1] + ir[2], _y = i * ir[4] + ir[5], _w = i * ir[7] + ir[8];
        for (int j = 0; j < w; ++j, _x += ir[0], _y += ir[3], _w += ir[6]) {
            const double ww = 1. / _w, x = _x * ww, y = _y * ww;
            const double x2 = x * x, y2 = y * y;
            const double r2 = x2 + y2, _2xy = 2 * x * y;
            const double kr = (1 + ((k3 * r2 + k2) * r2 + k1) * r2) / (1 + ((k6 * r2 + k5) * r2 + k4) * r2);
            const double u = fx * (x * kr + p1 * _2xy + p2 * (r2 + 2 * x2)) + u0;
            const double v = fy * (y * kr + p1 * (r2 + 2 * y2) + p2 * _2xy) + v0;
            const double us = u * 32, vs = v * 32;          /* saturate_cast<int> = cvRound (lrint, round half to even) */
            const int iu = us >= 2147483647.0 ? INT32_MAX : us <= -2147483648.0 ? INT32_MIN : (int)std::lrint(us);
            const int iv = vs >= 2147483647.0 ? INT32_MAX : vs <= -2147483648.0 ? INT32_MIN : (int)std::lrint(vs);
            const size_t o = (size_t)i * w + j;
            map_xy[2 * o] = (int16_t)(iu >> 5);
            map_xy[2 * o + 1] = (int16_t)(iv >> 5);
            map_frac[o] = (uint16_t)((iv & 31) * 32 + (iu & 31));
        }
    }
}

/* cv::remap(src, dst, map (CV_16SC2), INTER_LINEAR, BORDER_CONSTANT, 0) on u8, imgproc/imgwarp.cpp remapBilinear with
 * FixedPtCast<int, uchar, INTER_REMAP_COEF_BITS = 15>: BilinearTab_i weights (32-a)(32-b)*32, a(32-b)*32, (32-a)b*32, ab*32;
 * a tap outside the source reads the border value 0.  dst has the map's size. */
void ellc_oracle_remap_u8(const uint8_t* src, int sw, int sh, const int16_t* map_xy, const uint16_t* map_frac, int w, int h, uint8_t* dst) {
    for (int i = 0; i < h; ++i)
        for (int j = 0; j < w; ++j) {
            const size_t o = (size_t)i * w + j;
            const int x0 = map_xy[2 * o], y0 = map_xy[2 * o + 1], a = map_frac[o] & 31, b = (map_frac[o] >> 5) & 31;
            int v[4];
            for (int k = 0; k < 4; ++k) {
                const int xx = x0 + (k & 1), yy = y0 + (k >> 1);
                v[k] = (xx >= 0 && xx < sw && yy >= 0 && yy < sh) ? src[(size_t)yy * sw + xx] : 0;
            }
            const int s = v[0] * (32 - a) * (32 - b) * 32 + v[1] * a * (32 - b) * 32 + v[2] * (32 - a) * b * 32 + v[3] * a * b * 32;
            dst[o] = (uint8_t)std::min(std::max((s + (1 << 14)) >> 15, 0), 255);
        }
}

/* cv::resize(src, dst, Size(dw, dh), 0, 0, INTER_LINEAR) on u8, imgproc/imgwarp.cpp resize() generic branch:
 * inv_scale = dsize / ssize, scale = 1 / inv_scale; fx = (float)((dx + 0.5) * scale - 0.5), sx = cvFloor(fx), fx -= sx, clamped at
 * both borders; ialpha = saturate_cast<short>(cbuf * 2048); HResizeLinear (int sums), then VResizeLinear<uchar, int, short> as
 * VResizeLinearVec_32s8u computes it.  (dsize = ssize / 2 exactly takes the INTER_AREA branch there; its (a+b+c+d+2) >> 2 is
 * what these tables give at scale 2, coefficients 1024 / 1024.) */
static void oracle_resize_axis(int ssize, int dsize, std::vector<int>& ofs, std::vector<int>& ofs1, std::vector<int>& c0, std::vector<int>& c1) {
    const double inv_scale = (double)dsize / ssize, scale = 1. / inv_scale;
    ofs.resize(dsize); ofs1.resize(dsize); c0.resize(dsize); c1.resize(dsize);
    for (int d = 0; d < dsize; ++d) {
        float fx = (float)((d + 0.5) * scale - 0.5);
        int sx = (int)std::floor(fx);
        fx -= sx;
        if (sx < 0) { fx = 0; sx = 0; }
        if (sx + 1 >= ssize) { if (sx >= ssize - 1) { fx = 0; sx = ssize - 1; } }
        ofs[d] = sx; ofs1[d] = std::min(sx + 1, ssize - 1);
        const float cb0 = 1.f - fx, cb1 = fx;
        c0[d] = (int)std::lrint(cb0 * 2048); c1[d] = (int)std::lrint(cb1 * 2048);
    }
}
void ellc_oracle_resize_u8(const uint8_t* src, int sw, int sh, uint8_t* dst, int dw, int dh) {
    std::vector<int> xo, xo1, a0, a1, yo, yo1, b0, b1;
    oracle_resize_axis(sw, dw, xo, xo1, a0, a1);
    oracle_resize_axis(sh, dh, yo, yo1, b0, b1);
    std::vector<int> hbuf((size_t)sh * dw);
    for (int y = 0; y < sh; ++y)
        for (int x = 0; x < dw; ++x)
            hbuf[(size_t)y * dw + x] = src[(size_t)y * sw + xo[x]] * a0[x] + src[(size_t)y * sw + xo1[x]] * a1[x];
    for (int y = 0; y < dh; ++y)
        for (int x = 0; x < dw; ++x) {
            const int h0 = hbuf[(size_t)yo[y] * dw + x], h1 = hbuf[(size_t)yo1[y] * dw + x];
            const int v = (((b0[y] * (h0 >> 4)) >> 16) + ((b1[y] * (h1 >> 4)) >> 16) + 2) >> 2;
            dst[(size_t)y * dw + x] = (uint8_t)std::min(std::max(v, 0), 255);
        }
}

/* The whole step in the reference's order (SURVEY 3.1): gray, undistort (if set), resize to dw x dh. */
void ellc_oracle_ingest(const uint8_t* src, int w, int h, int channels, int pitch, int undistort, const double K[9], const double dist[5],
                        const double new_K[9], uint8_t* dst, int dw, int dh) {
    std::vector<uint8_t> gray((size_t)w * h), und;
    ellc_oracle_bgr2gray(src, w, h, channels, pitch, gray.data());
    const uint8_t* s = gray.data();
    if (undistort) {
        std::vector<int16_t> xy((size_t)2 * w * h);
        std::vector<uint16_t> fr((size_t)w * h);
        ellc_oracle_undistort_map(K, dist, new_K, w, h, xy.data(), fr.data());
        und.resize((size_t)w * h);
        ellc_oracle_remap_u8(gray.data(), w, h, xy.data(), fr.data(), w, h, und.data());
        s = und.data();
    }
    ellc_oracle_resize_u8(s, w, h, dst, dw, dh);
}

/* cv::getOptimalNewCameraMatrix(K, dist, size, alpha), centerPrincipalPoint = false, newImgSize = imgSize, as current OpenCV
 * computes it (calib3d getUndistortRectangles): a 9x9 double grid over the pixel centres 0 .. size-1 is undistorted by
 * undistortPoints (5 fixed-point iterations, normalised output); the inscribed and circumscribed rectangles give the projections
 * (size-1)/rect that map them onto the image, interpolated by alpha.  (OpenCV 3.0.0's icvGetRectangles sampled a float grid;
 * DESIGN.md section 9.) */
void ellc_oracle_optimal_new_camera_matrix(const double K[9], const double dist[5], int w, int h, double alpha, double new_K[9]) {
    const int N = 9;
    double px[N * N], py[N * N];
    for (int y = 0, k = 0; y < N; y++)
        for (int x = 0; x < N; x++) { px[k] = (double)x * (w - 1) / (N - 1); py[k] = (double)y * (h - 1) / (N - 1); k++; }
    const double fx = K[0], fy = K[4], ifx = 1. / fx, ify = 1. / fy, cx = K[2], cy = K[5];
    double k[8] = {dist[0], dist[1], dist[2], dist[3], dist[4], 0, 0, 0};
    for (int i = 0; i < N * N; i++) {
        double x = px[i], y = py[i], x0, y0;
        x0 = x = (x - cx) * ifx;
        y0 = y = (y - cy) * ify;
        for (int j = 0; j < 5; j++) {
            double r2 = x * x + y * y;
            double icdist = (1 + ((k[7] * r2 + k[6]) * r2 + k[5]) * r2) / (1 + ((k[4] * r2 + k[1]) * r2 + k[0]) * r2);
            if (icdist < 0) { x = x0; y = y0; break; }
            double deltaX = 2 * k[2] * x * y + k[3] * (r2 + 2 * x * x);
            double deltaY = k[2] * (r2 + 2 * y * y) + 2 * k[3] * x * y;
            x = (x0 - deltaX) * icdist;
            y = (y0 - deltaY) * icdist;
        }
        px[i] = x; py[i] = y;
    }
    double iX0 = -FLT_MAX, iX1 = FLT_MAX, iY0 = -FLT_MAX, iY1 = FLT_MAX, oX0 = FLT_MAX, oX1 = -FLT_MAX, oY0 = FLT_MAX, oY1 = -FLT_MAX;
    for (int y = 0, i = 0; y < N; y++)
        for (int x = 0; x < N; x++, i++) {
            oX0 = std::min(oX0, px[i]); oX1 = std::max(oX1, px[i]); oY0 = std::min(oY0, py[i]); oY1 = std::max(oY1, py[i]);
            if (x == 0) iX0 = std::max(iX0, px[i]);
            if (x == N - 1) iX1 = std::min(iX1, px[i]);
            if (y == 0) iY0 = std::max(iY0, py[i]);
            if (y == N - 1) iY1 = std::min(iY1, py[i]);
        }
    const double inner[4] = {iX0, iY0, iX1 - iX0, iY1 - iY0}, outer[4] = {oX0, oY0, oX1 - oX0, oY1 - oY0};
    const double fx0 = (w - 1) / inner[2], fy0 = (h - 1) / inner[3], cx0 = -fx0 * inner[0], cy0 = -fy0 * inner[1];
    const double fx1 = (w - 1) / outer[2], fy1 = (h - 1) / outer[3], cx1 = -fx1 * outer[0], cy1 = -fy1 * outer[1];
    for (int i = 0; i < 9; ++i) new_K[i] = K[i];
    new_K[0] = fx0 * (1 - alpha) + fx1 * alpha;
    new_K[4] = fy0 * (1 - alpha) + fy1 * alpha;
    new_K[2] = cx0 * (1 - alpha) + cx1 * alpha;
    new_K[5] = cy0 * (1 - alpha) + cy1 * alpha;
}

}  // extern "C"
