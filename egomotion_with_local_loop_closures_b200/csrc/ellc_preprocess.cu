// ellc_preprocess.cu -- per-frame and per-keyframe preparation kernels (sm_100a).
//
//   K1  pyrdown_u8_kernel   frame::constructImagePyramids -> cv::pyrDown x3      (src/Frame.cpp:170-182)
//   K2  pack_tex_kernel     frame::calculateGradient for every level            (src/Frame.cpp:185-285), fused with the
//                           intensity into one 32-bit texel per pixel (ellc_common.cuh) so that a bilinear tap of the GN
//                           kernel is a single gather
//   K3  select_*_kernel     frame::calculateNonZeroDepthPts: mask = depth > 0, count (src/Frame.cpp:295-301), plus an
//                           order-preserving compaction of the selected pixels into SelGeo/SelPix lists (raster order)
//
// All kernels are batched over slots (blockIdx.z / blockIdx.y) so that a whole batch of frames costs 4 launches.
#include "ellc_internal.h"
#include "ellc_lie.cuh"

namespace ellc {

// BORDER_REFLECT_101 with repeated folding for tiny images
__device__ __forceinline__ int reflect101(int i, int n) {
    if (n == 1) return 0;
    while (i < 0 || i >= n) i = (i < 0) ? -i : 2 * n - 2 - i;
    return i;
}

// ------------------------------------------------------------------------------------------------------------------
// K1: one pyrDown step for a batch of slots.  32x8 output tile per CTA; the (67 x 19) source footprint is staged in
// shared memory, filtered horizontally into int rows, then vertically; out = (sum + 128) >> 8 (exact integer).
// ------------------------------------------------------------------------------------------------------------------
constexpr int PD_TX = 32, PD_TY = 8;
constexpr int PD_SW = 2 * PD_TX + 3, PD_SH = 2 * PD_TY + 3;

__global__ void __launch_bounds__(PD_TX * PD_TY)
pyrdown_u8_kernel(uint8_t* __restrict__ pool, int64_t slot_stride, const int* __restrict__ slots,
                  int64_t src_off, int sw, int sh, int64_t dst_off, int dw, int dh) {
    __shared__ uint8_t s_src[PD_SH][PD_SW + 1];
    __shared__ int s_row[PD_SH][PD_TX];
    uint8_t* base = pool + (int64_t)slots[blockIdx.z] * slot_stride;
    const uint8_t* __restrict__ src = base + src_off;
    uint8_t* __restrict__ dst = base + dst_off;
    const int ox = blockIdx.x * PD_TX, oy = blockIdx.y * PD_TY;
    const int tid = threadIdx.y * PD_TX + threadIdx.x;
    const int sx0 = 2 * ox - 2, sy0 = 2 * oy - 2;
    for (int i = tid; i < PD_SW * PD_SH; i += PD_TX * PD_TY) {
        const int ly = i / PD_SW, lx = i - ly * PD_SW;
        const int gy = reflect101(sy0 + ly, sh), gx = reflect101(sx0 + lx, sw);
        s_src[ly][lx] = src[(int64_t)gy * sw + gx];
    }
    __syncthreads();
    for (int i = tid; i < PD_SH * PD_TX; i += PD_TX * PD_TY) {
        const int ly = i / PD_TX, lx = i - ly * PD_TX;
        const uint8_t* r = &s_src[ly][2 * lx];
        s_row[ly][lx] = r[0] + 4 * r[1] + 6 * r[2] + 4 * r[3] + r[4];
    }
    __syncthreads();
    const int x = ox + threadIdx.x, y = oy + threadIdx.y;
    if (x < dw && y < dh) {
        const int ly = 2 * threadIdx.y, lx = threadIdx.x;
        const int acc = s_row[ly][lx] + 4 * s_row[ly + 1][lx] + 6 * s_row[ly + 2][lx] + 4 * s_row[ly + 3][lx] + s_row[ly + 4][lx];
        dst[(int64_t)y * dw + x] = (uint8_t)((acc + 128) >> 8);
    }
}

// Word-wide form of K1 for source widths that are a multiple of 8 (all BASELINE sizes).  One thread produces a strip of
// 4 (x) by PDV_R (y) output pixels: per source row it loads 4 aligned words (its 8 bytes plus the neighbours' halo), forms
// the four horizontal [1 4 6 4 1] sums in registers, and keeps a five-row sliding window of them for the vertical pass;
// adjacent threads own adjacent output quads, so loads and the 4-byte stores are coalesced.  Same exact integer result.
constexpr int PDV_R = 8;
__device__ __forceinline__ void pdv_hrow(const uint8_t* __restrict__ row, int cq, int last_cq, int (&h)[4]) {
    const uint2 ab = *reinterpret_cast<const uint2*>(row + 8 * cq);
    uint32_t l, r;
    if (cq == 0) l = __byte_perm(ab.x, 0, 0x1200);               // reflect-101: bytes -2, -1 = bytes 2, 1 (placed at positions 2, 3)
    else l = *reinterpret_cast<const uint32_t*>(row + 8 * cq - 4);
    if (cq == last_cq) r = __byte_perm(ab.y, 0, 0x4012);         // bytes w, w+1, w+2 = bytes w-2, w-3, w-4
    else r = *reinterpret_cast<const uint32_t*>(row + 8 * cq + 8);
    int sb[13];
    sb[0] = (l >> 16) & 0xff; sb[1] = l >> 24;
#pragma unroll
    for (int i = 0; i < 4; ++i) { sb[2 + i] = (ab.x >> (8 * i)) & 0xff; sb[6 + i] = (ab.y >> (8 * i)) & 0xff; }
    sb[10] = r & 0xff; sb[11] = (r >> 8) & 0xff; sb[12] = (r >> 16) & 0xff;
#pragma unroll
    for (int j = 0; j < 4; ++j) h[j] = sb[2 * j] + 4 * sb[2 * j + 1] + 6 * sb[2 * j + 2] + 4 * sb[2 * j + 3] + sb[2 * j + 4];
}

__global__ void __launch_bounds__(128)
pyrdown_u8_vec_kernel(uint8_t* __restrict__ pool, int64_t slot_stride, const int* __restrict__ slots,
                      int64_t src_off, int sw, int sh, int64_t dst_off, int dw, int dh) {
    const int dwq = dw >> 2;                                     // output quads per row
    const int item = blockIdx.x * blockDim.x + threadIdx.x;
    const int strips = (dh + PDV_R - 1) / PDV_R;
    if (item >= dwq * strips) return;
    const int cq = item % dwq, y0 = (item / dwq) * PDV_R;
    uint8_t* base = pool + (int64_t)slots[blockIdx.y] * slot_stride;
    const uint8_t* __restrict__ src = base + src_off;
    uint8_t* __restrict__ dst = base + dst_off;
    int h[5][4];
#pragma unroll
    for (int k = 0; k < 3; ++k) pdv_hrow(src + (int64_t)reflect101(2 * y0 - 2 + k, sh) * sw, cq, dwq - 1, h[k]);
#pragma unroll
    for (int i = 0; i < PDV_R; ++i) {
        const int y = y0 + i;
        if (y >= dh) break;
        pdv_hrow(src + (int64_t)reflect101(2 * y + 1, sh) * sw, cq, dwq - 1, h[3]);
        pdv_hrow(src + (int64_t)reflect101(2 * y + 2, sh) * sw, cq, dwq - 1, h[4]);
        uint32_t o = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int acc = h[0][j] + 4 * h[1][j] + 6 * h[2][j] + 4 * h[3][j] + h[4][j];
            o |= (uint32_t)((acc + 128) >> 8) << (8 * j);
        }
        *reinterpret_cast<uint32_t*>(dst + (int64_t)y * dw + 4 * cq) = o;
#pragma unroll
        for (int j = 0; j < 4; ++j) { h[0][j] = h[2][j]; h[1][j] = h[3][j]; h[2][j] = h[4][j]; }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// K2: packed texels for all levels of a batch of frame slots.  One thread per pixel of the concatenated level windows.
// Border rule of src/Frame.cpp:222-283: one-sided, un-halved differences on the 1-px border of the (cols x rows) window.
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
pack_tex_kernel(const uint8_t* __restrict__ img_pool, int64_t img_slot_stride, uint32_t* __restrict__ tex_pool,
                int64_t tex_slot_stride, const int* __restrict__ slots, Geometry geo) {
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= geo.win_off[kLevels]) return;
    if (gid < kTexPad) tex_pool[(int64_t)slots[blockIdx.y] * tex_slot_stride + gid] = kTexZero;   // the out-of-bounds texel
    int level = 0;
#pragma unroll
    for (int l = 1; l < kLevels; ++l) level += (gid >= geo.win_off[l]);
    const int cols = geo.cols[level], rows = geo.rows[level], stride = geo.pyr_w[level];
    const int local = (int)(gid - geo.win_off[level]);
    const int y = local / cols, x = local - y * cols;
    const int slot = slots[blockIdx.y];
    const uint8_t* __restrict__ img = img_pool + (int64_t)slot * img_slot_stride + geo.img_off[level];
    const uint8_t* r = img + (int64_t)y * stride;
    const int c = r[x];
    int gx2, gy2;
    if (x == 0) gx2 = 2 * ((int)r[1] - c);
    else if (x == cols - 1) gx2 = 2 * (c - (int)r[x - 1]);
    else gx2 = (int)r[x + 1] - (int)r[x - 1];
    if (y == 0) gy2 = 2 * ((int)r[stride + x] - c);
    else if (y == rows - 1) gy2 = 2 * (c - (int)r[x - stride]);
    else gy2 = (int)r[stride + x] - (int)r[x - stride];
    tex_pool[(int64_t)slot * tex_slot_stride + kTexPad + gid] = tex_pack(c, gx2, gy2);
}

// Vector form for pyramids whose every level has a multiple-of-4 width (all BASELINE sizes): one thread packs four
// consecutive texels -- three 32-bit row loads plus two neighbour bytes in, one 16-byte store out -- so the kernel streams
// at HBM speed (P bytes in, 4 P bytes out per frame) instead of issuing five byte loads per texel.
__global__ void __launch_bounds__(256)
pack_tex_vec4_kernel(const uint8_t* __restrict__ img_pool, int64_t img_slot_stride, uint32_t* __restrict__ tex_pool,
                     int64_t tex_slot_stride, const int* __restrict__ slots, Geometry geo) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;          // quad index over the concatenated windows
    if (q * 4 >= geo.win_off[kLevels]) return;
    const int slot = slots[blockIdx.y];
    uint32_t* __restrict__ tex = tex_pool + (int64_t)slot * tex_slot_stride;
    if (q == 0) *reinterpret_cast<uint4*>(tex) = make_uint4(kTexZero, kTexZero, kTexZero, kTexZero);   // the out-of-bounds texel
    const int64_t gid = q * 4;
    int level = 0;
#pragma unroll
    for (int l = 1; l < kLevels; ++l) level += (gid >= geo.win_off[l]);
    const int cols = geo.cols[level], rows = geo.rows[level], stride = geo.pyr_w[level];
    const int local = (int)(gid - geo.win_off[level]);
    const int y = local / cols, x0 = local - y * cols;
    const uint8_t* __restrict__ r = img_pool + (int64_t)slot * img_slot_stride + geo.img_off[level] + (int64_t)y * stride;
    const uint32_t cw = *reinterpret_cast<const uint32_t*>(r + x0);
    const bool top = (y == 0), bot = (y == rows - 1);
    const uint32_t uw = *reinterpret_cast<const uint32_t*>(r + x0 - (top ? 0 : stride));
    const uint32_t dw = *reinterpret_cast<const uint32_t*>(r + x0 + (bot ? 0 : stride));
    int c[6];                                               // I[x0-1 .. x0+4]
    c[1] = cw & 0xff; c[2] = (cw >> 8) & 0xff; c[3] = (cw >> 16) & 0xff; c[4] = cw >> 24;
    c[0] = (x0 > 0) ? r[x0 - 1] : 0;
    c[5] = (x0 + 4 < cols) ? r[x0 + 4] : 0;
    uint32_t out[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int x = x0 + i, ci = c[i + 1];
        const int up = (uw >> (8 * i)) & 0xff, dn = (dw >> (8 * i)) & 0xff;
        int gx2, gy2;
        if (x == 0) gx2 = 2 * (c[i + 2] - ci);
        else if (x == cols - 1) gx2 = 2 * (ci - c[i]);
        else gx2 = c[i + 2] - c[i];
        if (top) gy2 = 2 * (dn - ci);
        else if (bot) gy2 = 2 * (ci - up);
        else gy2 = dn - up;
        out[i] = tex_pack(ci, gx2, gy2);
    }
    *reinterpret_cast<uint4*>(tex + kTexPad + gid) = make_uint4(out[0], out[1], out[2], out[3]);
}

// ------------------------------------------------------------------------------------------------------------------
// K3: selection.  Pass A counts per row and writes the mask, pass B scans the row counts per level, pass C writes the
// compacted SelGeo/SelPix lists in raster order (deterministic).
// ------------------------------------------------------------------------------------------------------------------
constexpr int SEL_T = 128;

__device__ __forceinline__ void row_to_level(const Geometry& geo, int grow, int& level, int& y) {
    level = 0;
    int base = 0;
    bool open = true;
#pragma unroll
    for (int l = 0; l < kLevels - 1; ++l) {
        const int next = base + geo.rows[l];
        if (open && grow >= next) { base = next; level = l + 1; }
        else open = false;
    }
    y = grow - base;
}

__global__ void __launch_bounds__(SEL_T)
select_count_kernel(const float* __restrict__ depth_pool, int64_t win_slot_stride, uint8_t* __restrict__ mask_pool,
                    int* __restrict__ rowcount_pool, int rows_total, const int* __restrict__ slots, Geometry geo) {
    int level, y;
    row_to_level(geo, blockIdx.x, level, y);
    const int slot = slots[blockIdx.y];
    const int cols = geo.cols[level];
    const int64_t off = (int64_t)slot * win_slot_stride + geo.win_off[level] + (int64_t)y * cols;
    const float* __restrict__ d = depth_pool + off;
    uint8_t* __restrict__ m = mask_pool + off;
    int cnt = 0;
    for (int x = threadIdx.x; x < cols; x += SEL_T) {
        const bool sel = d[x] > 0.0f;             // NaN compares false -> unselected, as cv::compare
        m[x] = sel ? 255 : 0;
        cnt += sel;
    }
    __shared__ int s_w[SEL_T / 32];
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < SEL_T / 32; ++w) t += s_w[w];
        rowcount_pool[(int64_t)slot * rows_total + blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(1024)
select_scan_kernel(const int* __restrict__ rowcount_pool, int* __restrict__ rowoff_pool, int* __restrict__ count_pool,
                   int rows_total, const int* __restrict__ slots, Geometry geo) {
    const int level = blockIdx.x;
    const int slot = slots[blockIdx.y];
    int base = 0;
    for (int l = 0; l < level; ++l) base += geo.rows[l];
    const int rows = geo.rows[level];
    const int* __restrict__ rc = rowcount_pool + (int64_t)slot * rows_total + base;
    int* __restrict__ ro = rowoff_pool + (int64_t)slot * rows_total + base;
    __shared__ int s_warp[32];
    __shared__ int s_carry;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int start = 0; start < rows; start += 1024) {
        const int i = start + threadIdx.x;
        const int v = (i < rows) ? rc[i] : 0;
        int inc = v;
        for (int o = 1; o < 32; o <<= 1) {
            const int n = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += n;
        }
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            int w = s_warp[lane];
            for (int o = 1; o < 32; o <<= 1) {
                const int n = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += n;
            }
            s_warp[lane] = w;                      // inclusive scan of warp totals
        }
        __syncthreads();
        const int carry = s_carry;
        const int wbase = (warp == 0) ? 0 : s_warp[warp - 1];
        if (i < rows) ro[i] = carry + wbase + inc - v;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = carry + s_warp[31];
        __syncthreads();
    }
    if (threadIdx.x == 0) count_pool[slot * kLevels + level] = s_carry;
}

struct KSet { LevelK k[kLevels]; };

__global__ void __launch_bounds__(SEL_T)
select_write_kernel(const float* __restrict__ depth_pool, const float* __restrict__ var_pool, int64_t win_slot_stride,
                    const uint8_t* __restrict__ img_pool, int64_t img_slot_stride, const int* __restrict__ rowoff_pool,
                    int rows_total, SelGeo* __restrict__ geo_pool, SelPix* __restrict__ pix_pool,
                    float* __restrict__ ikf_pool, KSet ks,
                    const int* __restrict__ slots, Geometry geo) {
    int level, y;
    row_to_level(geo, blockIdx.x, level, y);
    const int slot = slots[blockIdx.y];
    const int cols = geo.cols[level];
    const LevelK K = ks.k[level];
    const int64_t off = (int64_t)slot * win_slot_stride + geo.win_off[level] + (int64_t)y * cols;
    const float* __restrict__ d = depth_pool + off;
    const float* __restrict__ v = var_pool + off;
    const uint8_t* __restrict__ img = img_pool + (int64_t)slot * img_slot_stride + geo.img_off[level] + (int64_t)y * geo.pyr_w[level];
    const int64_t obase = (int64_t)slot * win_slot_stride + geo.win_off[level] + rowoff_pool[(int64_t)slot * rows_total + blockIdx.x];
    SelGeo* __restrict__ og = geo_pool + obase;
    SelPix* __restrict__ op = pix_pool + obase;
    float* __restrict__ ok = ikf_pool + obase;
    // worldpointY's numerator factor (y - cy) is row-constant
    const float yc = __fsub_rn((float)y, K.cy);
    __shared__ int s_w[SEL_T / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int running = 0;
    for (int start = 0; start < cols; start += SEL_T) {
        const int x = start + threadIdx.x;
        float dep = 0.f;
        bool sel = false;
        if (x < cols) { dep = d[x]; sel = dep > 0.0f; }
        const unsigned bal = __ballot_sync(0xffffffffu, sel);
        const int rank_in_warp = __popc(bal & ((1u << lane) - 1u));
        if (lane == 0) s_w[warp] = __popc(bal);
        __syncthreads();
        int wbase = 0, total = 0;
#pragma unroll
        for (int w = 0; w < SEL_T / 32; ++w) {
            const int c = s_w[w];
            if (w < warp) wbase += c;
            total += c;
        }
        if (sel) {
            SelGeo g;
            // src/PixelWisePyramid.cpp:236-237: (x - cx) * depth / fx, each operation rounded to fp32
            g.wX = __fdiv_rn(__fmul_rn(__fsub_rn((float)x, K.cx), dep), K.fx);
            g.wY = __fdiv_rn(__fmul_rn(yc, dep), K.fy);
            g.depth = dep;
            g.var = v[x];
            const int o = running + wbase + rank_in_warp;
            og[o] = g;
            op[o] = selpix_pack(x, y, img[x]);
            ok[o] = 8388608.0f + (float)img[x];           // 2^23 + I_kf: same float format as the kernel's intensity taps
        }
        running += total;
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Keyframe weight pyramid and loop-closure records (the constant-weight variant, src/PixelWisePyramid.cpp:500-680, :938).
// ------------------------------------------------------------------------------------------------------------------
// saveWeights(true), :546-548: weight_pyramid[level] += display_weightimg, once per tracked frame, in the caller's frame
// order (fp32, so the order is part of the result).  display_weightimg is zero where the mask is (:209-221); the frame
// slot's weight image is only written at selected pixels, so the keyframe's mask supplies the zeros.
__global__ void __launch_bounds__(256)
accumulate_weights_kernel(float* __restrict__ kf_w, const uint8_t* __restrict__ mask, const float* __restrict__ frw_pool,
                          int64_t win, const int* __restrict__ frame_slots, int n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= win) return;
    float w = kf_w[i];
    const bool sel = mask[i] != 0;
    for (int f = 0; f < n; ++f) w = __fadd_rn(w, sel ? frw_pool[(int64_t)frame_slots[f] * win + i] : 0.0f);
    kf_w[i] = w;
}

// frame::finaliseWeights, src/Frame.cpp:678-695: weight_pyramid[level] = weight_pyramid[level] / numWeightsAdded[level] when it
// is > 0.  cv::Mat / scalar multiplies by the reciprocal (MatOp_AddEx with alpha = 1./s, applied in float), it does not divide.
struct Counts4 { int c[kLevels]; };
__global__ void __launch_bounds__(256) finalise_weights_kernel(float* __restrict__ kf_w, Counts4 cnt, Geometry geo) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= geo.win_off[kLevels]) return;
    int level = 0;
#pragma unroll
    for (int l = 1; l < kLevels; ++l) level += (i >= geo.win_off[l]);
    if (cnt.c[level] > 0) kf_w[i] = __fmul_rn(kf_w[i], (float)(1.0 / (double)cnt.c[level]));
}

// precomputePixelWiseInvCompositional (:561-680) for the selected pixels of one keyframe level, in selection-list order, plus
// hessian = weightedSteepestDescent * steepestDescent^T (:938).  cv::gemm on CV_32F accumulates the float x float products in
// double and rounds once, so the sum is taken in double here too (the order of a double sum of ~1e5 float products does not
// reach the fp32 result).  One CTA per (level, keyframe); the Jacobian follows the reference's operation sequence exactly
// (fp32, with the sub-expressions C++ promotes to double through pow()).
// REF (ELLC_ARITH_REFERENCE): the reference's own order instead of the tree -- thread a*6+b sums (double)(J_a w) * (double)J_b over
// the level's records in raster order, one double addition after the other from +0 (the products are exact), and rounds once.
template <bool REF>
__global__ void __launch_bounds__(256)
lc_prepare_kernel(const SelGeo* __restrict__ geo_pool, const SelPix* __restrict__ pix_pool, int64_t rec_slot_stride,
                  const int* __restrict__ count_pool, const uint8_t* __restrict__ img_pool, int64_t img_slot_stride,
                  const float* __restrict__ weight_pool, LcRec* __restrict__ lc_pool, float4* __restrict__ lcf_pool,
                  uint32_t* __restrict__ lcp_pool, float* __restrict__ lc_H, KSet ks, const int* __restrict__ slots, Geometry geo) {
    const int level = blockIdx.x, slot = slots[blockIdx.y];
    const LevelK K = ks.k[level];
    const int cols = geo.cols[level], rows = geo.rows[level], stride = geo.pyr_w[level];
    const int n = count_pool[slot * kLevels + level];
    const int64_t rec_off = (int64_t)slot * rec_slot_stride + geo.win_off[level];
    const uint8_t* __restrict__ img = img_pool + (int64_t)slot * img_slot_stride + geo.img_off[level];
    const float* __restrict__ wimg = weight_pool + (int64_t)slot * geo.win_off[kLevels] + geo.win_off[level];
    double Hd[36];
#pragma unroll
    for (int i = 0; i < 36; ++i) Hd[i] = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const SelPix px = pix_pool[rec_off + i];
        const int x = selpix_x(px), y = selpix_y(px);
        const SelGeo sg = geo_pool[rec_off + i];
        const float dep = sg.depth;
        // prev_frame->gradientx/y at (x, y): frame::calculateGradient, src/Frame.cpp:185-285
        const uint8_t* r = img + (int64_t)y * stride;
        const int c = r[x];
        int gx2, gy2;
        if (x == 0) gx2 = 2 * ((int)r[1] - c);
        else if (x == cols - 1) gx2 = 2 * (c - (int)r[x - 1]);
        else gx2 = (int)r[x + 1] - (int)r[x - 1];
        if (y == 0) gy2 = 2 * ((int)r[stride + x] - c);
        else if (y == rows - 1) gy2 = 2 * (c - (int)r[x - stride]);
        else gy2 = (int)r[stride + x] - (int)r[x - stride];
        const float gradx = 0.5f * (float)gx2, grady = 0.5f * (float)gy2;
        // :639-666
        const float xc = __fsub_rn((float)x, K.cx), yc = __fsub_rn((float)y, K.cy);
        const double dfx = K.fx, dfy = K.fy, dgx = gradx, dgy = grady, dxc = xc, dyc = yc;
        const double idep = __ddiv_rn(1.0, (double)dep);
        const float jb0 = (float)__dmul_rn(dgy, -__dadd_rn(dfy, __ddiv_rn(__dmul_rn(dyc, dyc), dfy)));
        const float jt0 = __fmul_rn(gradx, __fdiv_rn(-__fmul_rn(yc, xc), K.fy));
        const float jb1 = __fmul_rn(grady, __fdiv_rn(__fmul_rn(yc, xc), K.fx));
        const float jt1 = (float)__dmul_rn(dgx, __dadd_rn(dfx, __ddiv_rn(__dmul_rn(dxc, dxc), dfx)));
        const float jb2 = __fmul_rn(grady, __fdiv_rn(__fmul_rn(K.fy, xc), K.fx));
        const float jt2 = __fmul_rn(gradx, -__fdiv_rn(__fmul_rn(K.fx, yc), K.fy));
        const float jt3 = (float)__dmul_rn(dgx, __dmul_rn(dfx, idep));
        const float jb4 = (float)__dmul_rn(dgy, __dmul_rn(dfy, idep));
        const float jb5 = (float)__dmul_rn(dgy, __dmul_rn(-dyc, idep));
        const float jt5 = (float)__dmul_rn(dgx, __dmul_rn(-dxc, idep));
        LcRec rec;
        rec.J[0] = __fadd_rn(jt0, jb0); rec.J[1] = __fadd_rn(jt1, jb1); rec.J[2] = __fadd_rn(jt2, jb2);
        rec.J[3] = __fadd_rn(jt3, 0.f); rec.J[4] = __fadd_rn(0.f, jb4); rec.J[5] = __fadd_rn(jt5, jb5);
        rec.w = wimg[y * cols + x];                                                    // weight_pyramid[level] :668
        rec.pad = 0.f;
        lc_pool[rec_off + i] = rec;
        // FAST flavour: 20 bytes instead of 52 -- the iteration rebuilds J from the keyframe pixel's gradients (kept exactly, as a
        // texel word in the frame texel format) and the back-projected point; the loop-closure kernel streams these records from
        // DRAM every iteration (the records of the resident keyframes are far larger than L2)
        lcf_pool[rec_off + i] = make_float4(sg.wX, sg.wY, sg.depth, rec.w);
        lcp_pool[rec_off + i] = (uint32_t)(gx2 + 512) | ((uint32_t)(gy2 + 512) << 10) | ((uint32_t)c << 24);
        if constexpr (!REF) {
#pragma unroll
            for (int a = 0; a < 6; ++a) {
                const double wj = (double)__fmul_rn(rec.J[a], rec.w);                  // weightedSteepestDescent :668-673
#pragma unroll
                for (int b = 0; b < 6; ++b) Hd[a * 6 + b] = fma(wj, (double)rec.J[b], Hd[a * 6 + b]);
            }
        }
    }
    __shared__ double s_part[8][36];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if constexpr (!REF) {
#pragma unroll
        for (int i = 0; i < 36; ++i) {
            double v = Hd[i];
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0) s_part[warp][i] = v;
        }
    }
    __syncthreads();                                                                   // (REF: the level's records are written)
    __shared__ float s_H[36];
    float* const rec = lc_H + ((int64_t)slot * kLevels + level) * kLcHStride;
    if (threadIdx.x < 36) {
        double t;
        if constexpr (REF) {
            const int a = threadIdx.x / 6, b = threadIdx.x % 6;
            const LcRec* lr = lc_pool + rec_off;
            t = 0.0;
#pragma unroll 4
            for (int i = 0; i < n; ++i) t = __dadd_rn(t, __dmul_rn((double)__fmul_rn(lr[i].J[a], lr[i].w), (double)lr[i].J[b]));
        } else {
            t = s_part[0][threadIdx.x];
            for (int w = 1; w < 8; ++w) t += s_part[w][threadIdx.x];
        }
        s_H[threadIdx.x] = (float)t;
        rec[threadIdx.x] = (float)t;
    }
    __syncthreads();
    // hessianInv = hessian.inv() is taken ONCE per level by the reference too (iter == 0, :939): store it with the hessian, so
    // that an iteration of the loop-closure tracker starts at deltapose = -(hessianInv sd_param) without a 6x6 LU
    if (threadIdx.x == 0) {
        float H[36], Hinv[36];
#pragma unroll
        for (int i = 0; i < 36; ++i) H[i] = s_H[i];
        const bool ok = invert6_lu_f(H, Hinv);
#pragma unroll
        for (int i = 0; i < 36; ++i) rec[36 + i] = Hinv[i];
        rec[72] = ok ? 1.f : 0.f;
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Keyframe depth / variance pyramids from the depth module's per-pixel hypotheses (SURVEY 8f row 2): the step right before
// the tracker, so that a keyframe costs one 9-byte-per-pixel upload instead of two 4-level f32 pyramids.
// ------------------------------------------------------------------------------------------------------------------
// depthMap::updateDepthImage, src/DepthPropagation.cpp:1273-1300, fused with calculate_no_of_Seeds (:1804-1830, counted on the
// flags as they arrive).  Level 0 in the Mat convention (depth 0 = invalid, variance -1): buildInvVarDepth only reads a depth
// where the variance is positive, so it sees the same values as in the reference's -1 array.
__global__ void __launch_bounds__(256)
depth_from_hypotheses_kernel(const uint8_t* __restrict__ valid, const float* __restrict__ idepth, const float* __restrict__ var_s,
                             float* __restrict__ depth0, float* __restrict__ var0, uint8_t* __restrict__ valid_out,
                             int* __restrict__ n_valid, int w, int h) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    bool v = false;
    if (i < w * h) {
        const int y = i / w, x = i - y * w;
        v = valid[i] != 0;
        const bool inner = !(y < 3 || y >= h - 3 || x < 3 || x >= w - 3);
        const bool keep = v && inner;
        const float id = idepth[i];
        if (keep && id >= -0.05f) { depth0[i] = __fdiv_rn(1.0f, id); var0[i] = var_s[i]; }
        else { depth0[i] = 0.0f; var0[i] = -1.0f; }
        if (valid_out) valid_out[i] = keep ? 1 : 0;
    }
    const unsigned bal = __ballot_sync(0xffffffffu, v);
    if ((threadIdx.x & 31) == 0 && bal) atomicAdd(n_valid, __popc(bal));
}

// depthMap::buildInvVarDepth, src/DepthPropagation.cpp:1637-1719: one level from the previous one; the four children are
// accumulated in the reference's order with individually rounded fp32 operations.
__global__ void __launch_bounds__(256)
build_inv_var_depth_kernel(const float* __restrict__ ds, const float* __restrict__ vs, float* __restrict__ dd, float* __restrict__ vd,
                           int width, int height) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= width * height) return;
    const int y = i / width, x = i - y * width, sw = 2 * width;
    const int idx = 2 * (x + y * sw);
    const int off[4] = {0, 1, sw, sw + 1};
    float idepth_sum = 0.f, ivar_sum = 0.f;
    int num = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float var = vs[idx + off[k]];
        if (var > 0) {
            const float ivar = __fdiv_rn(1.0f, var);
            ivar_sum = __fadd_rn(ivar_sum, ivar);
            idepth_sum = __fadd_rn(idepth_sum, __fdiv_rn(__fmul_rn(ivar, 1.0f), ds[idx + off[k]]));   // ivar * 1.0f / depth
            ++num;
        }
    }
    if (num > 0) { dd[i] = __fdiv_rn(ivar_sum, idepth_sum); vd[i] = __fdiv_rn((float)num, ivar_sum); }
    else { dd[i] = 0.0f; vd[i] = -1.0f; }
}

// ------------------------------------------------------------------------------------------------------------------
// Loop-closure candidate gating (SURVEY 8f row 3): the per-frame histogram and the per-candidate statistics of
// globalOptimize::findMatch; the ring / window bookkeeping around them stays with the caller.
// ------------------------------------------------------------------------------------------------------------------
// calculateImageHistogram, src/GlobalOptimize.cpp:40-100.  Counts are integers (exact in fp32 up to 2^24 pixels), so the
// float sum and the normalisation are bit-identical to cv::calcHist + the reference's loops whatever the counting order.
__global__ void __launch_bounds__(256)
frame_histogram_kernel(const uint8_t* __restrict__ img_pool, int64_t img_slot_stride, const int* __restrict__ slots, int n_pixels,
                       float* __restrict__ hist_pool) {
    __shared__ unsigned s_cnt[256];
    const int slot = slots[blockIdx.x];
    const uint8_t* __restrict__ img = img_pool + (int64_t)slot * img_slot_stride;
    s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const int n4 = n_pixels >> 2;
    for (int i = threadIdx.x; i < n4; i += 256) {
        const uint32_t v = reinterpret_cast<const uint32_t*>(img)[i];
        atomicAdd(&s_cnt[v & 0xff], 1u); atomicAdd(&s_cnt[(v >> 8) & 0xff], 1u);
        atomicAdd(&s_cnt[(v >> 16) & 0xff], 1u); atomicAdd(&s_cnt[v >> 24], 1u);
    }
    for (int i = 4 * n4 + threadIdx.x; i < n_pixels; i += 256) atomicAdd(&s_cnt[img[i]], 1u);
    __syncthreads();
    __shared__ float s_sum;
    if (threadIdx.x == 0) {
        float sum = 0.f;
        for (int i = 0; i < 256; ++i) sum = __fadd_rn(sum, (float)s_cnt[i]);      // :78-83, sequential
        s_sum = sum;
    }
    __syncthreads();
    hist_pool[(int64_t)slot * 256 + threadIdx.x] = __fdiv_rn((float)s_cnt[threadIdx.x], s_sum);   // :85-88
}

// Small host payloads (slot lists, pair lists, schedules) are pulled from the pinned staging arena by the SMs instead of
// the copy engine: a cudaMemcpyAsync on the compute stream would queue in the one H2D engine behind the bulk image /
// depth uploads of the NEXT batch (copy stream) and stall this batch's kernels for the whole upload burst.
__global__ void pull_host_words_kernel(uint32_t* __restrict__ dst, const uint32_t* __restrict__ src_host, int n_words) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_words; i += gridDim.x * blockDim.x) dst[i] = src_host[i];
}

// ------------------------------------------------------------------------------------------------------------------
// launch wrappers
// ------------------------------------------------------------------------------------------------------------------
__global__ void fill_f32_kernel(float* __restrict__ dst, float value, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) dst[i] = value;
}
int launch_fill_f32(cudaStream_t st, float* dst, float value, int64_t n) {
    if (n <= 0) return 0;
    fill_f32_kernel<<<148, 256, 0, st>>>(dst, value, n);
    return 1;
}

int launch_pull_host(cudaStream_t st, void* dst, const void* src_host_devptr, size_t bytes) {
    const int n_words = (int)((bytes + 3) / 4);
    if (n_words <= 0) return 0;
    int blocks = (n_words + 255) / 256;
    if (blocks > 148) blocks = 148;
    pull_host_words_kernel<<<blocks, 256, 0, st>>>((uint32_t*)dst, (const uint32_t*)src_host_devptr, n_words);
    return 1;
}

int launch_pyramid(cudaStream_t st, uint8_t* img_pool, int64_t img_slot_stride, const int* d_slots, int n, const Geometry& geo) {
    int launches = 0;
    for (int l = 1; l < kLevels; ++l) {
        const int sw = geo.pyr_w[l - 1], sh = geo.pyr_h[l - 1], dw = geo.pyr_w[l], dh = geo.pyr_h[l];
        if (sw % 8 == 0 && sw >= 16 && sh >= 2 && img_slot_stride % 8 == 0 && geo.img_off[l - 1] % 8 == 0 && geo.img_off[l] % 4 == 0) {
            const int items = (dw / 4) * ((dh + PDV_R - 1) / PDV_R);
            pyrdown_u8_vec_kernel<<<dim3((items + 127) / 128, n), 128, 0, st>>>(img_pool, img_slot_stride, d_slots, geo.img_off[l - 1],
                                                                                sw, sh, geo.img_off[l], dw, dh);
        } else {
            dim3 grid((dw + PD_TX - 1) / PD_TX, (dh + PD_TY - 1) / PD_TY, n);
            pyrdown_u8_kernel<<<grid, dim3(PD_TX, PD_TY), 0, st>>>(img_pool, img_slot_stride, d_slots, geo.img_off[l - 1],
                                                                   sw, sh, geo.img_off[l], dw, dh);
        }
        ++launches;
    }
    return launches;
}

int launch_pack_tex(cudaStream_t st, const uint8_t* img_pool, int64_t img_slot_stride, uint32_t* tex_pool,
                    int64_t tex_slot_stride, const int* d_slots, int n, const Geometry& geo) {
    bool vec = (img_slot_stride % 4 == 0) && (tex_slot_stride % 4 == 0);
    for (int l = 0; l < kLevels; ++l)
        vec = vec && (geo.cols[l] % 4 == 0) && (geo.pyr_w[l] % 4 == 0) && (geo.img_off[l] % 4 == 0) && (geo.win_off[l] % 4 == 0);
    if (vec) {
        dim3 grid((unsigned)((geo.win_off[kLevels] / 4 + 255) / 256), n);
        pack_tex_vec4_kernel<<<grid, 256, 0, st>>>(img_pool, img_slot_stride, tex_pool, tex_slot_stride, d_slots, geo);
    } else {
        dim3 grid((unsigned)((geo.win_off[kLevels] + 255) / 256), n);
        pack_tex_kernel<<<grid, 256, 0, st>>>(img_pool, img_slot_stride, tex_pool, tex_slot_stride, d_slots, geo);
    }
    return 1;
}

int launch_select(cudaStream_t st, const float* depth_pool, const float* var_pool, int64_t win_slot_stride,
                  const uint8_t* img_pool, int64_t img_slot_stride, uint8_t* mask_pool, int* rowcount_pool,
                  int* rowoff_pool, int* count_pool, SelGeo* geo_pool, SelPix* pix_pool, float* ikf_pool, const LevelK* K,
                  const int* d_slots, int n, const Geometry& geo) {
    int rows_total = 0;
    for (int l = 0; l < kLevels; ++l) rows_total += geo.rows[l];
    select_count_kernel<<<dim3(rows_total, n), SEL_T, 0, st>>>(depth_pool, win_slot_stride, mask_pool, rowcount_pool,
                                                                rows_total, d_slots, geo);
    select_scan_kernel<<<dim3(kLevels, n), 1024, 0, st>>>(rowcount_pool, rowoff_pool, count_pool, rows_total, d_slots, geo);
    KSet ks;
    for (int l = 0; l < kLevels; ++l) ks.k[l] = K[l];
    select_write_kernel<<<dim3(rows_total, n), SEL_T, 0, st>>>(depth_pool, var_pool, win_slot_stride, img_pool,
                                                                img_slot_stride, rowoff_pool, rows_total, geo_pool,
                                                                pix_pool, ikf_pool, ks, d_slots, geo);
    return 3;
}

int launch_depth_pyramid(cudaStream_t st, const uint8_t* d_valid, const float* d_idepth, const float* d_var_s, float* depth_slot,
                         float* var_slot, uint8_t* d_valid_out, int* d_n_valid, const Geometry& geo) {
    const int w = geo.width, h = geo.height;
    depth_from_hypotheses_kernel<<<(w * h + 255) / 256, 256, 0, st>>>(d_valid, d_idepth, d_var_s, depth_slot, var_slot, d_valid_out, d_n_valid, w, h);
    for (int l = 1; l < kLevels; ++l) {
        const int n = geo.cols[l] * geo.rows[l];
        build_inv_var_depth_kernel<<<(n + 255) / 256, 256, 0, st>>>(depth_slot + geo.win_off[l - 1], var_slot + geo.win_off[l - 1],
                                                                    depth_slot + geo.win_off[l], var_slot + geo.win_off[l],
                                                                    geo.cols[l], geo.rows[l]);
    }
    return kLevels;
}

int launch_frame_histograms(cudaStream_t st, const uint8_t* img_pool, int64_t img_slot_stride, const int* d_slots, int n, int n_pixels,
                            float* hist_pool) {
    frame_histogram_kernel<<<n, 256, 0, st>>>(img_pool, img_slot_stride, d_slots, n_pixels, hist_pool);
    return 1;
}

int launch_accumulate_weights(cudaStream_t st, float* kf_weight_slot, const uint8_t* mask_slot, const float* frw_pool,
                              int64_t win, const int* d_frame_slots, int n) {
    accumulate_weights_kernel<<<(unsigned)((win + 255) / 256), 256, 0, st>>>(kf_weight_slot, mask_slot, frw_pool, win, d_frame_slots, n);
    return 1;
}

int launch_finalise_weights(cudaStream_t st, float* kf_weight_slot, const int counts[kLevels], const Geometry& geo) {
    Counts4 c;
    for (int l = 0; l < kLevels; ++l) c.c[l] = counts[l];
    finalise_weights_kernel<<<(unsigned)((geo.win_off[kLevels] + 255) / 256), 256, 0, st>>>(kf_weight_slot, c, geo);
    return 1;
}

int launch_lc_prepare(cudaStream_t st, const SelGeo* geo_pool, const SelPix* pix_pool, int64_t rec_slot_stride, const int* count_pool,
                      const uint8_t* img_pool, int64_t img_slot_stride, const float* weight_pool, LcRec* lc_pool, float4* lcf_pool,
                      uint32_t* lcp_pool, float* lc_H, const LevelK* K, const int* d_slots, int n, const Geometry& geo, bool reference) {
    KSet ks;
    for (int l = 0; l < kLevels; ++l) ks.k[l] = K[l];
    if (reference)
        lc_prepare_kernel<true><<<dim3(kLevels, n), 256, 0, st>>>(geo_pool, pix_pool, rec_slot_stride, count_pool, img_pool, img_slot_stride,
                                                                  weight_pool, lc_pool, lcf_pool, lcp_pool, lc_H, ks, d_slots, geo);
    else
        lc_prepare_kernel<false><<<dim3(kLevels, n), 256, 0, st>>>(geo_pool, pix_pool, rec_slot_stride, count_pool, img_pool, img_slot_stride,
                                                                   weight_pool, lc_pool, lcf_pool, lcp_pool, lc_H, ks, d_slots, geo);
    return 1;
}

}  // namespace ellc
