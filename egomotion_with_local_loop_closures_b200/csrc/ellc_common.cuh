// ellc_common.cuh -- shared device/host types of the B200 GN tracker (internal; the public ABI is include/ellc_gn.h).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/ellc_gn.h"

namespace ellc {

constexpr int kLevels = ELLC_LEVELS;
constexpr int kLcHStride = 80;              // floats per (keyframe, level) record of the loop-closure hessian: H, H^-1, ok, pad

// One selected keyframe pixel (mask != 0, src/Frame.cpp:298), produced once per keyframe level by the selection
// kernels and streamed by every GN iteration as two coalesced loads (16 B + 4 B, structure of arrays).
//   SelGeo: the back-projected point of src/PixelWisePyramid.cpp:236-238 -- it depends only on the keyframe pixel, its
//           depth and the intrinsics, so it is evaluated once (with the reference's exact fp32 operation sequence)
//           instead of in every iteration -- plus the depth variance of :348.
//   SelPix: x | y << 11 | I_kf << 22   (x, y < 2048; I_kf = prev_frame->image_pyramid[level](y,x), :189)
struct __align__(16) SelGeo {
    float wX, wY;       // worldpointX / worldpointY
    float depth;        // worldpointZ = depth_ptr[x]
    float var;          // currentDepthMap->depthvararrptr[level][idx]
};
static_assert(sizeof(SelGeo) == 16, "SelGeo must be 16 bytes");
typedef uint32_t SelPix;
__host__ __device__ inline SelPix selpix_pack(int x, int y, int ikf) { return (uint32_t)x | ((uint32_t)y << 11) | ((uint32_t)ikf << 22); }
__host__ __device__ inline int selpix_x(SelPix p) { return (int)(p & 0x7ffu); }
__host__ __device__ inline int selpix_y(SelPix p) { return (int)((p >> 11) & 0x7ffu); }
__host__ __device__ inline int selpix_i(SelPix p) { return (int)(p >> 22); }

// Packed texel of the current frame at one pyramid level: everything one bilinear tap needs in one 32-bit word.
//   bits  0.. 9  2*gradx + 512   (gradx of src/Frame.cpp:185-285 is a multiple of 0.5 in [-255, 255])
//   bits 10..19  2*grady + 512
//   bits 24..31  intensity I
// The biased fields sit inside the mantissa range of a float, so the GN kernel turns each of them into an exact float
// with ONE logic instruction ((t & mask) | magic exponent, PRMT for the intensity byte) instead of shift + mask +
// int->float conversion.  Interpolating the doubled integer gradients and halving is bit-identical to interpolating the
// reference's f32 gradient maps (scaling by 2 is exact).  kTexZero is an out-of-bounds tap (pixVal = 0,
// src/Frame.h:211-215): I = 0, gradx = grady = 0.
__host__ __device__ inline uint32_t tex_pack(int I, int gx2, int gy2) {
    return (uint32_t)(gx2 + 512) | ((uint32_t)(gy2 + 512) << 10) | ((uint32_t)I << 24);
}
constexpr uint32_t kTexZero = 512u | (512u << 10);
constexpr int kTexPad = 4;      // words reserved at the start of every frame slot of the texel pool; they hold kTexZero
constexpr int kTexTail = 4096;  // mapped words behind the last slot (weight-0 taps may read one row past a level)
__host__ __device__ inline int tex_I(uint32_t w) { return (int)(w >> 24); }
__host__ __device__ inline int tex_gx2(uint32_t w) { return (int)(w & 0x3ffu) - 512; }
__host__ __device__ inline int tex_gy2(uint32_t w) { return (int)((w >> 10) & 0x3ffu) - 512; }
constexpr int kRecTail = 8192;

// Loop-closure (inverse-compositional, constant-weight) record of one selected keyframe pixel, built once per keyframe by
// lc_prepare_kernel: the steepest-descent row of src/PixelWisePyramid.cpp:633-666 (keyframe gradients at the keyframe
// pixel: it does not depend on the pose) and the keyframe's finalised weight (weight_pyramid[level], :668).
struct __align__(16) LcRec {
    float J[6];
    float w;
    float pad;
};
static_assert(sizeof(LcRec) == 32, "LcRec must be 32 bytes");  // mapped records behind the last keyframe slot (the pixel loop prefetches past a level's end)

// Geometry of the pyramid for one configuration.
struct Geometry {
    int width, height;
    int pyr_w[kLevels], pyr_h[kLevels];        // cv::pyrDown dims: ceil-halving (image_pyramid[l])
    int cols[kLevels], rows[kLevels];          // currentCols/currentRows = width>>l, height>>l (src/Frame.cpp:321-322)
    int64_t img_off[kLevels + 1];              // element offsets of the u8 pyramid levels inside a slot
    int64_t win_off[kLevels + 1];              // element offsets of (cols x rows) level arrays (depth/var/mask/tex/recs)
};

// Per-level intrinsics, GetIntrinsic (src/UserDefinedFunc.cpp:33-49)
struct LevelK {
    float fx, fy, cx, cy;
    float ifx, ify;            // fast-mode reciprocals
    float fy_ifx, fx_ify;      // fy/fx, fx/fy
    float cm1, rm1;            // float(cols-1), float(rows-1): nCols / nRows of src/Frame.h:196-197
    // bit patterns of float(cols), float(cols-1), float(rows), float(rows-1): for a projected coordinate u that is not
    // -0.0, (u >= 0 && floor(u) <= cols-1) == (bits(u) < bits(float(cols))) and (u >= 0 && u <= cols-1) ==
    // (bits(u) <= bits(float(cols-1))) as unsigned compares (negative and NaN patterns are larger than any bound)
    uint32_t colsf_bits, cm1_bits, rowsf_bits, rm1_bits;
};

struct TrackParams {
    Geometry geo;
    LevelK K[kLevels];
    int max_iter[kLevels];
    float huber_half;          // HUBER_D / 2
    float noise2;              // CAMERA_PIXEL_NOISE_2
    float weight[6];
    float stop_threshold;
    int jacobian_at_warped;
    // pools
    const uint32_t* tex_pool;  int64_t tex_slot_stride;       // packed texels, per frame slot
    const SelGeo* geo_pool;    int64_t rec_slot_stride;       // selection records, per keyframe slot
    const SelPix* pix_pool;
    const float* ikf_pool;                                    // 2^23 + I_kf per selected pixel (fast flavour)
    const int* count_pool;                                    // [kf_slot][kLevels]
    // work
    const ellc_pair* pairs;
    const int* order;          // optional schedule: CTA cluster c tracks pairs[order[c]]
    ellc_result* results;
    ellc_iter_trace* trace;    // optional [pair][level][ELLC_MAX_TRACE_ITERS]
    int n_pairs;
    int pairs_per_cta;         // pairs tracked in lockstep by one CTA (1..4); clusters always track one
    // evaluate-only mode (ellc_gn_evaluate): run `level_hi..level_lo`, `iter_limit` iterations, no pose update
    int level_hi, level_lo;
    int iter_limit;            // 0 = use max_iter
    int no_update;
    float* weight_out;         // optional display_weightimg of the evaluated level (cols x rows), evaluate-only mode
    float* frw_pool;           // per frame slot: display_weightimg of every level (win layout) for ELLC_PAIR_SAVE_WEIGHTS pairs
    const LcRec* lc_pool;      // loop-closure records, per keyframe slot (rec_slot_stride)
    const float4* lcf_pool;    // compact loop-closure records of the FAST flavour: {wX, wY, depth, weight} ...
    const uint32_t* lcp_pool;  // ... + the keyframe pixel as a texel word (2 gradx + 512 : 10 | 2 grady + 512 : 10 | - | I : 8): 20 B / pixel
    const float* lc_H;         // [kf_slot][kLevels][kLcHStride]: hessian (36, src/PixelWisePyramid.cpp:938), hessianInv (36, :939), ok (1)
    uint32_t zero_mask;        // always 0: an opaque zero the pixel loop uses to build ordering dependences
    float lm_lambda, lm_up, lm_down;   // Levenberg-Marquardt damping (0 = plain Gauss-Newton, the reference) and its step-rejection factors
    // multi-GPU result exchange (ellc_track_batch_exchange): besides `results`, the record of pair i is stored at
    // xchg_dst[d][xchg_index[i]] for d < xchg_n -- result tables in the memory of this or of peer GPUs (NVLink stores)
    // display planes of the evaluated level (STRICT flavour, evaluate mode): 4 planes of cols x rows floats --
    // display_warpedimg, display_iterationres, savedWarpedPointsX, savedWarpedPointsY (src/PixelWisePyramid.cpp:262-283, :332)
    float* disp_out;
    int xchg_n;
    ellc_result* xchg_dst[ELLC_MAX_RANKS];
    const int* xchg_index;
    // ELLC_ARITH_REFERENCE: the per-row record offsets of the selection lists ([kf_slot][rows_total], rows of the levels
    // concatenated; select_scan_kernel), from which the row bands of the reference's summation become record ranges, and the
    // number of row bands of the constant-weight variant (FLAG_DO_PARALLEL_CONST_WEIGHT_POSE_EST ? 2 : 1)
    const int* rowoff_pool;
    int rows_total;
    int lc_bands;
};

}  // namespace ellc
