// ellc_lie.cuh -- SE(3) pose algebra and the 6x6 solve, shared by the device kernels and the host-side pose helpers.
//
// Replaces (citations relative to the reference repo):
//   - Eigen .exp() on hat(pose)            src/PixelWisePyramid.cpp:153-159   -> the same published algorithm Eigen 3.2.5's
//                                             MatrixExponential<float> implements (Pade 3/5/7 by L1 norm + scaling and
//                                             squaring, fp32, individually rounded ops), so R|t carry the reference's rounding
//   - concatenateRelativePose               src/Frame.cpp:503-530             -> log(exp(a) exp(b)): fp32 Pade exps, fp32 4x4
//                                             product, exact SE(3) logarithm evaluated in double and rounded to fp32
//   - concatenateOriginPose                 src/Frame.cpp:534-562             -> log(exp(a) exp(b)^-1)
//   - cv::Mat::inv() (DECOMP_LU, CV_32F)    src/PixelWisePyramid.cpp:451      -> same partial-pivot LU in fp32, eps 10*FLT_EPSILON,
//                                                                               singular => all-zero inverse (zero step)
//   - updatePose()                          src/PixelWisePyramid.cpp:460-491
//
// Everything here runs once per GN iteration on ONE thread while the rest of the CTA waits, so it is written to stay in
// registers: fixed-size arrays, fully unrollable loops, and row swaps done with selects instead of dynamic indexing
// (the arithmetic and its order are unchanged by that).
#pragma once

#include <cuda_runtime.h>
#include <math.h>

namespace ellc {

#ifdef __CUDA_ARCH__
#define ELLC_MUL(a, b) __fmul_rn((a), (b))
#define ELLC_ADD(a, b) __fadd_rn((a), (b))
#define ELLC_SUB(a, b) __fsub_rn((a), (b))
#define ELLC_DIV(a, b) __fdiv_rn((a), (b))
#define ELLC_DMUL(a, b) __dmul_rn((a), (b))
#define ELLC_DADD(a, b) __dadd_rn((a), (b))
#define ELLC_UNROLL _Pragma("unroll")
#else
#define ELLC_MUL(a, b) ((a) * (b))
#define ELLC_ADD(a, b) ((a) + (b))
#define ELLC_SUB(a, b) ((a) - (b))
#define ELLC_DIV(a, b) ((a) / (b))
#define ELLC_DMUL(a, b) ((a) * (b))
#define ELLC_DADD(a, b) ((a) + (b))
#define ELLC_UNROLL
#endif

// log of a rigid transform (R row-major, t) -> 6-vector, in double.  Entry extraction as src/Frame.cpp:523-528:
// omega = theta/sin(theta) * (antisymmetric part), v = V^-1 t.  For rotations below ~17 degrees (everything this
// tracker produces) theta/sin(theta) and the V^-1 coefficient come from their power series (no atan2/sin/cos calls);
// both agree with the closed forms to ~1e-16, far inside the final rounding to fp32.
__host__ __device__ inline void se3_log_d(const double R[9], const double t[3], double out[6]) {
    const double ax = 0.5 * (R[7] - R[5]), ay = 0.5 * (R[2] - R[6]), az = 0.5 * (R[3] - R[1]);   // sin(th) n
    const double s2 = ax * ax + ay * ay + az * az;
    const double c = 0.5 * (R[0] + R[4] + R[8] - 1.0);
    double k, th2;
    if (c > 0.5 && s2 < 0.09 * c * c) {
        // th = atan(q), q = s/c; k = th/s = (atan(q)/q)/c; atan(q)/q = sum (-1)^n q^2n/(2n+1), |q| < 0.3
        const double q2 = s2 / (c * c);
        double p = 0.0;
        ELLC_UNROLL
        for (int n = 17; n >= 0; --n) p = p * q2 + ((n & 1) ? -1.0 : 1.0) / (double)(2 * n + 1);
        k = p / c;
        th2 = p * p * q2;                     // th^2 = (q p)^2
    } else {
        const double s = sqrt(s2);
        const double th = atan2(s, c);
        if (s < 1e-7) k = (c > 0) ? 1.0 + th * th / 6.0 : 0.0;
        else k = th / s;
        th2 = th * th;
    }
    const double w[3] = {k * ax, k * ay, k * az};
    double coef;                              // (1 - th sin th / (2 (1 - cos th))) / th^2
    if (th2 < 0.1) {
        coef = 1.0 / 12.0 + th2 * (1.0 / 720.0 + th2 * (1.0 / 30240.0 + th2 * (1.0 / 1209600.0 + th2 * (1.0 / 47900160.0 +
               th2 * (691.0 / 1307674368000.0)))));
    } else {
        const double th = sqrt(th2);
        coef = (1.0 - (th * sin(th)) / (2.0 * (1.0 - cos(th)))) / th2;
    }
    const double wt[3] = {w[1] * t[2] - w[2] * t[1], w[2] * t[0] - w[0] * t[2], w[0] * t[1] - w[1] * t[0]};
    const double wwt[3] = {w[1] * wt[2] - w[2] * wt[1], w[2] * wt[0] - w[0] * wt[2], w[0] * wt[1] - w[1] * wt[0]};
    out[0] = w[0]; out[1] = w[1]; out[2] = w[2];
    ELLC_UNROLL
    for (int i = 0; i < 3; ++i) out[3 + i] = t[i] - 0.5 * wt[i] + coef * wwt[i];
}

// ---- fp32 4x4 helpers (row-major), every operation individually rounded -------------------------------------------
__host__ __device__ inline void m4_mul_f(const float (&x)[16], const float (&y)[16], float (&r)[16]) {
    ELLC_UNROLL
    for (int i = 0; i < 4; ++i) {
        ELLC_UNROLL
        for (int j = 0; j < 4; ++j) {
            float s = ELLC_MUL(x[i * 4 + 0], y[0 * 4 + j]);
            ELLC_UNROLL
            for (int k = 1; k < 4; ++k) s = ELLC_ADD(s, ELLC_MUL(x[i * 4 + k], y[k * 4 + j]));
            r[i * 4 + j] = s;
        }
    }
}
// r = c2*P + c1*Q + c0*S + ci*I, left to right; NP = number of leading matrix operands used (1..3)
template <int NP>
__host__ __device__ inline void m4_poly_f(float c2, const float (&P)[16], float c1, const float (&Q)[16], float c0,
                                          const float (&S)[16], float ci, float (&r)[16]) {
    ELLC_UNROLL
    for (int i = 0; i < 16; ++i) {
        float s = ELLC_MUL(c2, P[i]);
        if (NP >= 2) s = ELLC_ADD(s, ELLC_MUL(c1, Q[i]));
        if (NP >= 3) s = ELLC_ADD(s, ELLC_MUL(c0, S[i]));
        r[i] = ELLC_ADD(s, (i % 5 == 0) ? ci : 0.f);
    }
}
// Solve A X = B for 4x4 fp32 with partial-pivot LU (the PartialPivLU::solve step of the Pade quotient, and .inverse()).
__host__ __device__ inline void lu4_solve_f(const float (&Ain)[16], const float (&Bin)[16], float (&X)[16]) {
    // (loops with constant bounds and the triangular condition inside: see invert6_lu_warp)
    constexpr int n = 4;
    float A[16], B[16];
    ELLC_UNROLL
    for (int i = 0; i < 16; ++i) { A[i] = Ain[i]; B[i] = Bin[i]; }
    ELLC_UNROLL
    for (int i = 0; i < n; ++i) {
        int p = i;
        float best = fabsf(A[i * n + i]);
        ELLC_UNROLL
        for (int r = 1; r < n; ++r) {
            if (r > i) {
                const float v = fabsf(A[r * n + i]);
                if (v > best) { best = v; p = r; }
            }
        }
        ELLC_UNROLL
        for (int r = 1; r < n; ++r) {                     // swap rows i and p (p is data dependent: select, don't index)
            if (r > i) {
                const bool sw = (p == r);
                ELLC_UNROLL
                for (int c = 0; c < n; ++c) {
                    const float a0 = A[i * n + c], a1 = A[r * n + c];
                    A[i * n + c] = sw ? a1 : a0; A[r * n + c] = sw ? a0 : a1;
                    const float b0 = B[i * n + c], b1 = B[r * n + c];
                    B[i * n + c] = sw ? b1 : b0; B[r * n + c] = sw ? b0 : b1;
                }
            }
        }
        const float piv = A[i * n + i];
        ELLC_UNROLL
        for (int r = 1; r < n; ++r) {
            if (r > i) {
                const float f = ELLC_DIV(A[r * n + i], piv);
                A[r * n + i] = f;
                ELLC_UNROLL
                for (int c = 1; c < n; ++c) if (c > i) A[r * n + c] = ELLC_SUB(A[r * n + c], ELLC_MUL(f, A[i * n + c]));
                ELLC_UNROLL
                for (int c = 0; c < n; ++c) B[r * n + c] = ELLC_SUB(B[r * n + c], ELLC_MUL(f, B[i * n + c]));
            }
        }
    }
    ELLC_UNROLL
    for (int c = 0; c < n; ++c) {
        ELLC_UNROLL
        for (int i = n - 1; i >= 0; --i) {
            float s = B[i * n + c];
            ELLC_UNROLL
            for (int k = 1; k < n; ++k) if (k > i) s = ELLC_SUB(s, ELLC_MUL(A[i * n + k], X[k * n + c]));
            X[i * n + c] = ELLC_DIV(s, A[i * n + i]);
        }
    }
}

// exp(hat(pose)) as a 4x4 fp32 matrix: Pade approximant chosen on the L1 norm (fp32 thresholds 0.42587 / 1.88015,
// scaling by 2^s above 3.92572), R = (V-U)^-1 (V+U), squared s times.
__host__ __device__ inline void se3_exp_pade_f(const float p[6], float (&T)[16]) {
    float M[16];
    ELLC_UNROLL
    for (int i = 0; i < 16; ++i) M[i] = 0.f;
    M[1] = -p[2]; M[2] = p[1];  M[3] = p[3];
    M[4] = p[2];  M[6] = -p[0]; M[7] = p[4];
    M[8] = -p[1]; M[9] = p[0];  M[11] = p[5];
    float l1 = 0.f;
    ELLC_UNROLL
    for (int j = 0; j < 4; ++j) {
        float s = 0.f;
        ELLC_UNROLL
        for (int i = 0; i < 4; ++i) s = ELLC_ADD(s, fabsf(M[i * 4 + j]));
        l1 = fmaxf(l1, s);
    }
    float U[16], V[16], A2[16], tmp[16];
    int squarings = 0;
    if (l1 < 4.258730016922831e-001f) {
        m4_mul_f(M, M, A2);
        m4_poly_f<1>(1.f, A2, 0.f, A2, 0.f, A2, 60.f, tmp);
        m4_mul_f(M, tmp, U);
        m4_poly_f<1>(12.f, A2, 0.f, A2, 0.f, A2, 120.f, V);
    } else if (l1 < 1.880152677804762e+000f) {
        float A4[16];
        m4_mul_f(M, M, A2);
        m4_mul_f(A2, A2, A4);
        m4_poly_f<2>(1.f, A4, 420.f, A2, 0.f, A2, 15120.f, tmp);
        m4_mul_f(M, tmp, U);
        m4_poly_f<2>(30.f, A4, 3360.f, A2, 0.f, A2, 30240.f, V);
    } else {
        float A[16], A4[16], A6[16];
        (void)frexpf(ELLC_DIV(l1, 3.925724783138660f), &squarings);
        if (squarings < 0) squarings = 0;
        const float sc = ldexpf(1.0f, squarings);
        ELLC_UNROLL
        for (int i = 0; i < 16; ++i) A[i] = ELLC_DIV(M[i], sc);
        m4_mul_f(A, A, A2);
        m4_mul_f(A2, A2, A4);
        m4_mul_f(A4, A2, A6);
        m4_poly_f<3>(1.f, A6, 1512.f, A4, 277200.f, A2, 8648640.f, tmp);
        m4_mul_f(A, tmp, U);
        m4_poly_f<3>(56.f, A6, 25200.f, A4, 1995840.f, A2, 17297280.f, V);
    }
    float num[16], den[16];
    ELLC_UNROLL
    for (int i = 0; i < 16; ++i) { num[i] = ELLC_ADD(U[i], V[i]); den[i] = ELLC_ADD(-U[i], V[i]); }
    lu4_solve_f(den, num, T);
    for (int s = 0; s < squarings; ++s) {
        m4_mul_f(T, T, tmp);
        ELLC_UNROLL
        for (int i = 0; i < 16; ++i) T[i] = tmp[i];
    }
}

// log of the rigid part of a 4x4 fp32 matrix -> fp32 6-vector (double evaluation, rounded once)
__host__ __device__ inline void m4_log_f(const float (&T)[16], float out[6]) {
    double R[9], t[3], o[6];
    ELLC_UNROLL
    for (int i = 0; i < 3; ++i) {
        ELLC_UNROLL
        for (int j = 0; j < 3; ++j) R[i * 3 + j] = (double)T[i * 4 + j];
        t[i] = (double)T[i * 4 + 3];
    }
    se3_log_d(R, t, o);
    ELLC_UNROLL
    for (int i = 0; i < 6; ++i) out[i] = (float)o[i];
}

// dest = log(exp(a) exp(b))   -- frame::concatenateRelativePose, src/Frame.cpp:503-530
__host__ __device__ inline void concat_relative_f(const float a[6], const float b[6], float dest[6]) {
    float Ta[16], Tb[16], T[16];
    se3_exp_pade_f(a, Ta);
    se3_exp_pade_f(b, Tb);
    m4_mul_f(Ta, Tb, T);
    m4_log_f(T, dest);
}

// dest = log(exp(a) exp(b)^-1) -- frame::concatenateOriginPose, src/Frame.cpp:534-562 (.inverse() = LU solve against I)
__host__ __device__ inline void concat_origin_f(const float a[6], const float b[6], float dest[6]) {
    float Ta[16], Tb[16], Ti[16], T[16], I[16];
    se3_exp_pade_f(a, Ta);
    se3_exp_pade_f(b, Tb);
    ELLC_UNROLL
    for (int i = 0; i < 16; ++i) I[i] = (i % 5 == 0) ? 1.f : 0.f;
    lu4_solve_f(Tb, I, Ti);
    m4_mul_f(Ta, Ti, T);
    m4_log_f(T, dest);
}

// exp(hat(pose)): SE3_vec[12] = r11 r12 r13 t1 r21 ... (src/PixelWisePyramid.cpp:162-173)
__host__ __device__ inline void pose_to_rt_f(const float pose[6], float Rt[12]) {
    float T[16];
    se3_exp_pade_f(pose, T);
    ELLC_UNROLL
    for (int i = 0; i < 12; ++i) Rt[i] = T[i];
}

// cv::Mat::inv() for a 6x6 CV_32F: partial-pivot LU on [A | I] in fp32 (each op individually rounded, as OpenCV's
// scalar LUImpl<float>), pivot threshold FLT_EPSILON*10, back-substitution multiplying by the stored reciprocal.
// Returns false and an all-zero inverse when singular (=> deltapose = 0, weightedPose = 0 < 1 => level ends).
__host__ __device__ inline bool invert6_lu_f(const float (&Hin)[36], float (&Hinv)[36]) {
    constexpr int m = 6;
    float A[36], B[36];
    ELLC_UNROLL
    for (int i = 0; i < 36; ++i) { A[i] = Hin[i]; B[i] = (i % 7 == 0) ? 1.f : 0.f; }
    const float eps = 1.1920929e-07f * 10;
    bool ok = true;
    ELLC_UNROLL
    for (int i = 0; i < m; ++i) {
        int k = i;
        float best = fabsf(A[i * m + i]);
        ELLC_UNROLL
        for (int j = 1; j < m; ++j) {
            if (j > i) {
                const float v = fabsf(A[j * m + i]);
                if (v > best) { best = v; k = j; }
            }
        }
        if (best < eps) ok = false;                           // LUImpl returns 0 here; keep going branch-free, zero below
        ELLC_UNROLL
        for (int j = 1; j < m; ++j) {                         // swap rows i and k: columns i.. of A, all of B
            if (j > i) {
                const bool sw = (k == j);
                ELLC_UNROLL
                for (int c = 0; c < m; ++c) {
                    if (c >= i) {
                        const float a0 = A[i * m + c], a1 = A[j * m + c];
                        A[i * m + c] = sw ? a1 : a0; A[j * m + c] = sw ? a0 : a1;
                    }
                }
                ELLC_UNROLL
                for (int c = 0; c < m; ++c) {
                    const float b0 = B[i * m + c], b1 = B[j * m + c];
                    B[i * m + c] = sw ? b1 : b0; B[j * m + c] = sw ? b0 : b1;
                }
            }
        }
        const float d = ELLC_DIV(-1.f, A[i * m + i]);
        ELLC_UNROLL
        for (int j = 1; j < m; ++j) {
            if (j > i) {
                const float alpha = ELLC_MUL(A[j * m + i], d);
                ELLC_UNROLL
                for (int c = 1; c < m; ++c) if (c > i) A[j * m + c] = ELLC_ADD(A[j * m + c], ELLC_MUL(alpha, A[i * m + c]));
                ELLC_UNROLL
                for (int c = 0; c < m; ++c) B[j * m + c] = ELLC_ADD(B[j * m + c], ELLC_MUL(alpha, B[i * m + c]));
            }
        }
        A[i * m + i] = -d;
    }
    ELLC_UNROLL
    for (int i = m - 1; i >= 0; --i) {
        ELLC_UNROLL
        for (int j = 0; j < m; ++j) {
            float s = B[i * m + j];
            ELLC_UNROLL
            for (int c = 1; c < m; ++c) if (c > i) s = ELLC_SUB(s, ELLC_MUL(A[i * m + c], B[c * m + j]));
            B[i * m + j] = ELLC_MUL(s, A[i * m + i]);
        }
    }
    ELLC_UNROLL
    for (int q = 0; q < 36; ++q) Hinv[q] = ok ? B[q] : 0.f;
    return ok;
}

// hessianInv = hessian.inv(); updatePose()  -- src/PixelWisePyramid.cpp:451-491.
// delta_i = -(sum_k Hinv[i][k] b[k]) with cv::gemm's double accumulator; weightedPose = sum |delta_i * weight_i|;
// pose <- log(exp(delta) exp(pose)).  Returns false if the hessian was singular.
__host__ __device__ inline bool solve_update_f(const float (&H)[36], const float (&b)[6], const float (&weight)[6],
                                               float (&pose)[6], float (&delta)[6], float* weighted_pose) {
    float Hinv[36];
    const bool ok = invert6_lu_f(H, Hinv);
    ELLC_UNROLL
    for (int i = 0; i < 6; ++i) {
        double s = 0.0;
        ELLC_UNROLL
        for (int k = 0; k < 6; ++k) s = ELLC_DADD(s, ELLC_DMUL((double)Hinv[i * 6 + k], (double)b[k]));
        delta[i] = -(float)s;
    }
    float wp = fabsf(ELLC_MUL(delta[0], weight[0]));
    ELLC_UNROLL
    for (int i = 1; i < 6; ++i) wp = ELLC_ADD(wp, fabsf(ELLC_MUL(delta[i], weight[i])));
    *weighted_pose = wp;
    float np[6];
    concat_relative_f(delta, pose, np);
    ELLC_UNROLL
    for (int i = 0; i < 6; ++i) pose[i] = np[i];
    return ok;
}


// ---- closed-form SE(3) exp / log for small rotations (FAST flavour of K5) -------------------------------------------------
// SURVEY 8a row I allows a closed-form replacement of Eigen's Pade exponential / Schur logarithm ("agrees to ~1e-6").  The FAST
// flavour of K5 uses these when every rotation involved is below kSmallTheta2 = 0.04 rad^2 (11.5 degrees: every pose a
// frame-to-keyframe track produces); anything larger takes the op-for-op Pade path, as does the STRICT flavour always.
// fp32 throughout, power series in theta^2 (truncation < 1e-10 at the bound), ~60 instructions each, no divisions:
// the Pade path costs ~700 per exponential even lane-distributed, and its 4x4 LU is a chain of 7 dependent divisions.
// Measured against the Pade / double-log path (tests/test_oracle_known_answers.py): entries of exp within 2.5e-7, log within 2e-7.
constexpr float kSmallTheta2 = 0.04f;

// exp(hat(p)), rows 0..2 (SE3_vec layout r11 r12 r13 t1 r21 ..., src/PixelWisePyramid.cpp:162-173); requires |omega|^2 < ~0.1
__host__ __device__ inline void se3_exp_small_f(const float p[6], float (&Rt)[12]) {
    const float wx = p[0], wy = p[1], wz = p[2], vx = p[3], vy = p[4], vz = p[5];
    const float t2 = wx * wx + wy * wy + wz * wz;
    // A = sin(t)/t, B = (1 - cos t)/t^2, C = (t - sin t)/t^3
    const float A = 1.0f - t2 * (1.0f / 6.0f) * (1.0f - t2 * (1.0f / 20.0f) * (1.0f - t2 * (1.0f / 42.0f) * (1.0f - t2 * (1.0f / 72.0f))));
    const float B = 0.5f * (1.0f - t2 * (1.0f / 12.0f) * (1.0f - t2 * (1.0f / 30.0f) * (1.0f - t2 * (1.0f / 56.0f) * (1.0f - t2 * (1.0f / 90.0f)))));
    const float C = (1.0f / 6.0f) * (1.0f - t2 * (1.0f / 20.0f) * (1.0f - t2 * (1.0f / 42.0f) * (1.0f - t2 * (1.0f / 72.0f) * (1.0f - t2 * (1.0f / 110.0f)))));
    // R = I + A W + B W^2, W^2 = w w^T - t2 I
    const float Bx = B * wx, By = B * wy, Bz = B * wz;
    const float d = 1.0f - B * t2;
    Rt[0] = d + Bx * wx;            Rt[1] = Bx * wy - A * wz;       Rt[2] = Bx * wz + A * wy;
    Rt[4] = Bx * wy + A * wz;       Rt[5] = d + By * wy;            Rt[6] = By * wz - A * wx;
    Rt[8] = Bx * wz - A * wy;       Rt[9] = By * wz + A * wx;       Rt[10] = d + Bz * wz;
    // t = V v, V = I + B W + C W^2:  v + B (w x v) + C (w x (w x v))
    const float cx = wy * vz - wz * vy, cy = wz * vx - wx * vz, cz = wx * vy - wy * vx;
    const float ex = wy * cz - wz * cy, ey = wz * cx - wx * cz, ez = wx * cy - wy * cx;
    Rt[3] = vx + B * cx + C * ex;
    Rt[7] = vy + B * cy + C * ey;
    Rt[11] = vz + B * cz + C * ez;
}

// log of the rigid transform in rows 0..2 of Rt -> pose, entry extraction as src/Frame.cpp:523-528.  Returns false (pose
// untouched) when the rotation is not small (sin^2 theta >= kSmallTheta2 or cos theta <= 0.9): the caller then takes the
// general path.  theta / sin(theta) from the arcsine series in sin^2 theta (of the antisymmetric part, exact differences for
// small rotations), V^-1 = I - W/2 + coef W^2 with coef = (1 - theta sin theta / (2 (1 - cos theta))) / theta^2 as a series.
__host__ __device__ inline bool se3_log_small_f(const float (&Rt)[12], float pose[6]) {
    const float ax = 0.5f * (Rt[9] - Rt[6]), ay = 0.5f * (Rt[2] - Rt[8]), az = 0.5f * (Rt[4] - Rt[1]);   // sin(theta) n
    const float s2 = ax * ax + ay * ay + az * az;
    const float c = 0.5f * (Rt[0] + Rt[5] + Rt[10] - 1.0f);
    if (!(s2 < kSmallTheta2 && c > 0.9f)) return false;
    // asin(s)/s = 1 + s2/6 + 3 s2^2/40 + 15 s2^3/336 + 105 s2^4/3456 + 945 s2^5/42240 + 10395 s2^6/599040
    const float k = 1.0f + s2 * (1.0f / 6.0f + s2 * (3.0f / 40.0f + s2 * (15.0f / 336.0f + s2 * (105.0f / 3456.0f +
                    s2 * (945.0f / 42240.0f + s2 * (10395.0f / 599040.0f))))));
    const float wx = k * ax, wy = k * ay, wz = k * az;
    const float t2 = (k * k) * s2;
    const float coef = 1.0f / 12.0f + t2 * (1.0f / 720.0f + t2 * (1.0f / 30240.0f + t2 * (1.0f / 1209600.0f)));
    const float tx = Rt[3], ty = Rt[7], tz = Rt[11];
    const float cx = wy * tz - wz * ty, cy = wz * tx - wx * tz, cz = wx * ty - wy * tx;
    const float ex = wy * cz - wz * cy, ey = wz * cx - wx * cz, ez = wx * cy - wy * cx;
    pose[0] = wx; pose[1] = wy; pose[2] = wz;
    pose[3] = tx - 0.5f * cx + coef * ex;
    pose[4] = ty - 0.5f * cy + coef * ey;
    pose[5] = tz - 0.5f * cz + coef * ez;
    return true;
}

// pose <- log(exp(delta) exp(pose)) with Rt = exp(hat(pose)) given and exp(hat(new pose)) returned: the FAST flavour's form of
// src/PixelWisePyramid.cpp:484 + :153-173.  Returns false (nothing written) when a rotation is too large for the series.
__host__ __device__ inline bool pose_update_small_f(const float (&delta)[6], const float (&Rt)[12], float (&pose)[6], float (&Rt_new)[12]) {
    const float td = delta[0] * delta[0] + delta[1] * delta[1] + delta[2] * delta[2];
    const float tp = pose[0] * pose[0] + pose[1] * pose[1] + pose[2] * pose[2];
    if (!(td < kSmallTheta2 && tp < kSmallTheta2)) return false;
    float E[12], T[12];
    se3_exp_small_f(delta, E);
    ELLC_UNROLL
    for (int i = 0; i < 3; ++i) {
        ELLC_UNROLL
        for (int j = 0; j < 4; ++j) {
            float s = E[4 * i] * Rt[j] + E[4 * i + 1] * Rt[4 + j] + E[4 * i + 2] * Rt[8 + j];
            if (j == 3) s += E[4 * i + 3];
            T[4 * i + j] = s;
        }
    }
    float np[6];
    if (!se3_log_small_f(T, np)) return false;
    ELLC_UNROLL
    for (int i = 0; i < 6; ++i) pose[i] = np[i];
    se3_exp_small_f(np, Rt_new);
    return true;
}

#ifdef __CUDACC__
// ---- warp-cooperative K5 (device only) -------------------------------------------------------------------------------
// The same LU as invert6_lu_f, with the six right-hand-side columns of [A | I] spread over lanes (lane % 6 owns one column
// of the inverse) while every lane eliminates A redundantly: identical pivots, identical operations per entry, 1/4 of the
// serial instruction count.  Returns column (lane % 6) of the inverse in col[0..5]; *ok as invert6_lu_f.
// All loops have constant bounds with the triangular condition inside: written as `for (j = i + 1; ...)` nvcc leaves the row
// loops rolled after unrolling the outer one, and A then lives in local memory with dynamic addressing (LDL/STL chains).
__device__ inline void invert6_lu_warp(const float (&Hin)[36], int lane, float (&col)[6], bool* okp) {
    constexpr int m = 6;
    const int mycol = lane % 6;
    float A[36], B[6];
    ELLC_UNROLL
    for (int i = 0; i < 36; ++i) A[i] = Hin[i];
    ELLC_UNROLL
    for (int i = 0; i < 6; ++i) B[i] = (i == mycol) ? 1.f : 0.f;
    const float eps = 1.1920929e-07f * 10;
    bool ok = true;
    ELLC_UNROLL
    for (int i = 0; i < m; ++i) {
        int k = i;
        float best = fabsf(A[i * m + i]);
        ELLC_UNROLL
        for (int j = 1; j < m; ++j) {
            if (j > i) {
                const float v = fabsf(A[j * m + i]);
                if (v > best) { best = v; k = j; }
            }
        }
        if (best < eps) ok = false;
        if (k != i) {                                          // warp-uniform (A is replicated); usually the diagonal is the pivot
            ELLC_UNROLL
            for (int j = 1; j < m; ++j) {
                if (j > i) {
                    const bool sw = (k == j);
                    ELLC_UNROLL
                    for (int c = 0; c < m; ++c) {
                        if (c >= i) {
                            const float a0 = A[i * m + c], a1 = A[j * m + c];
                            A[i * m + c] = sw ? a1 : a0; A[j * m + c] = sw ? a0 : a1;
                        }
                    }
                    const float b0 = B[i], b1 = B[j];
                    B[i] = sw ? b1 : b0; B[j] = sw ? b0 : b1;
                }
            }
        }
        const float d = ELLC_DIV(-1.f, A[i * m + i]);
        ELLC_UNROLL
        for (int j = 1; j < m; ++j) {
            if (j > i) {
                const float alpha = ELLC_MUL(A[j * m + i], d);
                ELLC_UNROLL
                for (int c = 1; c < m; ++c) if (c > i) A[j * m + c] = ELLC_ADD(A[j * m + c], ELLC_MUL(alpha, A[i * m + c]));
                B[j] = ELLC_ADD(B[j], ELLC_MUL(alpha, B[i]));
            }
        }
        A[i * m + i] = -d;
    }
    ELLC_UNROLL
    for (int i = m - 1; i >= 0; --i) {
        float s = B[i];
        ELLC_UNROLL
        for (int c = 1; c < m; ++c) if (c > i) s = ELLC_SUB(s, ELLC_MUL(A[i * m + c], B[c]));
        B[i] = ELLC_MUL(s, A[i * m + i]);
    }
    ELLC_UNROLL
    for (int q = 0; q < 6; ++q) col[q] = ok ? B[q] : 0.f;
    *okp = ok;
}

// ---- 4x4 fp32 algebra spread over the lanes of a warp ----------------------------------------------------------------
// Lane l holds entry e = l & 15 (row e >> 2, column e & 3) of every matrix; lanes 16..31 mirror lanes 0..15.  Each entry is
// produced by exactly the operation sequence of the serial helpers above (m4_mul_f, m4_poly_f, lu4_solve_f, se3_exp_pade_f),
// so the results are bit-identical to them; only who computes which entry changes.  A 4x4 product costs 8 shuffles + 7
// arithmetic instructions per lane instead of 112 on one thread, the Pade quotient 7 divisions instead of 22.
constexpr unsigned kFullWarp = 0xffffffffu;
__device__ __forceinline__ float m4w_mul(float x, float y, int e) {
    const int r4 = e & 12, c = e & 3;
    float s = ELLC_MUL(__shfl_sync(kFullWarp, x, r4), __shfl_sync(kFullWarp, y, c));
    ELLC_UNROLL
    for (int k = 1; k < 4; ++k) s = ELLC_ADD(s, ELLC_MUL(__shfl_sync(kFullWarp, x, r4 + k), __shfl_sync(kFullWarp, y, 4 * k + c)));
    return s;
}
// lu4_solve_f: entry e of X with A X = B
__device__ __forceinline__ float lu4w_solve(float A, float B, int e) {
    const int r = e >> 2, c = e & 3;
    ELLC_UNROLL
    for (int i = 0; i < 3; ++i) {                              // step i = 3 of the serial loop has nothing left to do
        int p = i;
        float best = fabsf(__shfl_sync(kFullWarp, A, 4 * i + i));
        ELLC_UNROLL
        for (int j = i + 1; j < 4; ++j) {
            const float v = fabsf(__shfl_sync(kFullWarp, A, 4 * j + i));
            if (v > best) { best = v; p = j; }
        }
        if (p != i) {                                          // warp-uniform: every lane saw the same column
            const int sr = (r == i) ? p : (r == p) ? i : r;
            A = __shfl_sync(kFullWarp, A, 4 * sr + c);
            B = __shfl_sync(kFullWarp, B, 4 * sr + c);
        }
        const float piv = __shfl_sync(kFullWarp, A, 5 * i);
        const float ari = __shfl_sync(kFullWarp, A, 4 * r + i);
        const float ai = __shfl_sync(kFullWarp, A, 4 * i + c);
        const float bi = __shfl_sync(kFullWarp, B, 4 * i + c);
        if (r > i) {
            const float f = ELLC_DIV(ari, piv);
            if (c > i) A = ELLC_SUB(A, ELLC_MUL(f, ai));
            else if (c == i) A = f;
            B = ELLC_SUB(B, ELLC_MUL(f, bi));
        }
    }
    const float d = __shfl_sync(kFullWarp, A, 5 * r);
    const float a1 = __shfl_sync(kFullWarp, A, 4 * r + 1), a2 = __shfl_sync(kFullWarp, A, 4 * r + 2),
                a3 = __shfl_sync(kFullWarp, A, 4 * r + 3);
    float X = ELLC_DIV(B, d);                                  // final for row 3
    const float x3 = __shfl_sync(kFullWarp, X, 12 + c);
    if (r == 2) X = ELLC_DIV(ELLC_SUB(B, ELLC_MUL(a3, x3)), d);
    const float x2 = __shfl_sync(kFullWarp, X, 8 + c);
    if (r == 1) X = ELLC_DIV(ELLC_SUB(ELLC_SUB(B, ELLC_MUL(a2, x2)), ELLC_MUL(a3, x3)), d);
    const float x1 = __shfl_sync(kFullWarp, X, 4 + c);
    if (r == 0) X = ELLC_DIV(ELLC_SUB(ELLC_SUB(ELLC_SUB(B, ELLC_MUL(a1, x1)), ELLC_MUL(a2, x2)), ELLC_MUL(a3, x3)), d);
    return X;
}
// se3_exp_pade_f: entry e of exp(hat(p)); p is the same in every lane.  Not inlined: K5 calls it twice per iteration and the
// solver's code should stay small (it runs on one warp per CTA and misses in the instruction cache otherwise).
static __device__ __noinline__ float se3_exp_pade_warp(float p0, float p1, float p2, float p3, float p4, float p5, int e) {
    const float p[6] = {p0, p1, p2, p3, p4, p5};          // by value: an array reference would put the caller's pose in local memory
    float M = 0.f;
    M = (e == 1) ? -p[2] : M; M = (e == 2) ? p[1] : M;  M = (e == 3) ? p[3] : M;
    M = (e == 4) ? p[2] : M;  M = (e == 6) ? -p[0] : M; M = (e == 7) ? p[4] : M;
    M = (e == 8) ? -p[1] : M; M = (e == 9) ? p[0] : M;  M = (e == 11) ? p[5] : M;
    // L1 norm: column sums in the serial order (the zero entries add exactly nothing)
    const float a0 = fabsf(p[0]), a1 = fabsf(p[1]), a2 = fabsf(p[2]);
    float l1 = fmaxf(0.f, ELLC_ADD(a2, a1));
    l1 = fmaxf(l1, ELLC_ADD(a2, a0));
    l1 = fmaxf(l1, ELLC_ADD(a1, a0));
    l1 = fmaxf(l1, ELLC_ADD(ELLC_ADD(fabsf(p[3]), fabsf(p[4])), fabsf(p[5])));
    const bool diag = (e % 5) == 0;
    float U, V;
    int squarings = 0;
    if (l1 < 4.258730016922831e-001f) {
        const float A2 = m4w_mul(M, M, e);
        const float tmp = ELLC_ADD(ELLC_MUL(1.f, A2), diag ? 60.f : 0.f);
        U = m4w_mul(M, tmp, e);
        V = ELLC_ADD(ELLC_MUL(12.f, A2), diag ? 120.f : 0.f);
    } else if (l1 < 1.880152677804762e+000f) {
        const float A2 = m4w_mul(M, M, e);
        const float A4 = m4w_mul(A2, A2, e);
        const float tmp = ELLC_ADD(ELLC_ADD(ELLC_MUL(1.f, A4), ELLC_MUL(420.f, A2)), diag ? 15120.f : 0.f);
        U = m4w_mul(M, tmp, e);
        V = ELLC_ADD(ELLC_ADD(ELLC_MUL(30.f, A4), ELLC_MUL(3360.f, A2)), diag ? 30240.f : 0.f);
    } else {
        (void)frexpf(ELLC_DIV(l1, 3.925724783138660f), &squarings);
        if (squarings < 0) squarings = 0;
        const float sc = ldexpf(1.0f, squarings);
        const float A = ELLC_DIV(M, sc);
        const float A2 = m4w_mul(A, A, e);
        const float A4 = m4w_mul(A2, A2, e);
        const float A6 = m4w_mul(A4, A2, e);
        const float tmp = ELLC_ADD(ELLC_ADD(ELLC_ADD(ELLC_MUL(1.f, A6), ELLC_MUL(1512.f, A4)), ELLC_MUL(277200.f, A2)),
                                   diag ? 8648640.f : 0.f);
        U = m4w_mul(A, tmp, e);
        V = ELLC_ADD(ELLC_ADD(ELLC_ADD(ELLC_MUL(56.f, A6), ELLC_MUL(25200.f, A4)), ELLC_MUL(1995840.f, A2)),
                     diag ? 17297280.f : 0.f);
    }
    float T = lu4w_solve(ELLC_ADD(-U, V), ELLC_ADD(U, V), e);
    for (int s = 0; s < squarings; ++s) T = m4w_mul(T, T, e);
    return T;
}

// solve_update_f executed by one full warp (all 32 lanes call it with the same H, b, weight, pose and get the same pose, delta,
// weighted_pose).  The 4x4 part runs lane-distributed: rt_pose_e is entry (lane & 15) of exp(hat(pose)) as computed for the
// current iteration (rows 0..2 from Rt, row 3 exactly [0 0 0 1]), and *rt_new_e returns the same entry of exp(hat(new pose)) for
// the next iteration (src/PixelWisePyramid.cpp:153-173), so only exp(delta) and exp(new pose) are evaluated.
// deltapose and weightedPose (:466-479) given column (lane % 6) of hessianInv in col[0..5] (all zeros for a singular hessian)
__device__ inline void delta_from_inverse_warp(const float (&col)[6], const float (&b)[6], const float (&weight)[6],
                                               float (&delta)[6], float* weighted_pose, int lane) {
    // delta_i = -(sum_k Hinv[i][k] b[k]): lane k (< 6) holds Hinv[.][k]; products are exact in double, the sum runs k = 0..5
    const double bk = (double)b[lane % 6];
    ELLC_UNROLL
    for (int i = 0; i < 6; ++i) {
        const double term = __dmul_rn((double)col[i], bk);
        double s = 0.0;
        ELLC_UNROLL
        for (int k = 0; k < 6; ++k) s = __dadd_rn(s, __shfl_sync(kFullWarp, term, k));
        delta[i] = -(float)s;
    }
    float wp = fabsf(ELLC_MUL(delta[0], weight[0]));
    ELLC_UNROLL
    for (int i = 1; i < 6; ++i) wp = ELLC_ADD(wp, fabsf(ELLC_MUL(delta[i], weight[i])));
    *weighted_pose = wp;
}
// The logarithm of ELLC_ARITH_REFERENCE: the closed form of the oracle's rigid_log (oracle/ellc_oracle.cpp:181-203) operation for
// operation -- every double operation individually rounded (no contraction), CUDA's double atan2 / sin / cos, the same
// s < 1e-7 and theta < 1e-4 branches -- where se3_log_d takes power series below ~17 degrees.  The two agree to ~1e-16 before the
// final rounding, but the closed form cancels at small angles (1 - cos theta), so only this one reproduces the reference's last
// float bit of the translation.
__device__ inline void m4_log_ref_f(const float (&T)[16], float out[6]) {
    const double R00 = T[0], R01 = T[1], R02 = T[2];
    const double R10 = T[4], R11 = T[5], R12 = T[6];
    const double R20 = T[8], R21 = T[9], R22 = T[10];
    const double t[3] = {T[3], T[7], T[11]};
    const double ax = __dmul_rn(0.5, __dsub_rn(R21, R12)), ay = __dmul_rn(0.5, __dsub_rn(R02, R20)), az = __dmul_rn(0.5, __dsub_rn(R10, R01));
    const double s = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(ax, ax), __dmul_rn(ay, ay)), __dmul_rn(az, az)));
    const double c = __dmul_rn(0.5, __dsub_rn(__dadd_rn(__dadd_rn(R00, R11), R22), 1.0));
    const double th = atan2(s, c);
    double k;
    if (s < 1e-7) k = (c > 0) ? __dadd_rn(1.0, __ddiv_rn(__dmul_rn(th, th), 6.0)) : 0.0;
    else k = __ddiv_rn(th, s);
    const double w[3] = {__dmul_rn(k, ax), __dmul_rn(k, ay), __dmul_rn(k, az)};
    double coef;
    if (th < 1e-4) coef = __dadd_rn(1.0 / 12.0, __ddiv_rn(__dmul_rn(th, th), 720.0));
    else coef = __ddiv_rn(__dsub_rn(1.0, __ddiv_rn(__dmul_rn(th, sin(th)), __dmul_rn(2.0, __dsub_rn(1.0, cos(th))))), __dmul_rn(th, th));
    const double wt[3] = {__dsub_rn(__dmul_rn(w[1], t[2]), __dmul_rn(w[2], t[1])), __dsub_rn(__dmul_rn(w[2], t[0]), __dmul_rn(w[0], t[2])),
                          __dsub_rn(__dmul_rn(w[0], t[1]), __dmul_rn(w[1], t[0]))};
    const double wwt[3] = {__dsub_rn(__dmul_rn(w[1], wt[2]), __dmul_rn(w[2], wt[1])), __dsub_rn(__dmul_rn(w[2], wt[0]), __dmul_rn(w[0], wt[2])),
                           __dsub_rn(__dmul_rn(w[0], wt[1]), __dmul_rn(w[1], wt[0]))};
    out[0] = (float)w[0]; out[1] = (float)w[1]; out[2] = (float)w[2];
    ELLC_UNROLL
    for (int i = 0; i < 3; ++i) out[3 + i] = (float)__dadd_rn(__dsub_rn(t[i], __dmul_rn(0.5, wt[i])), __dmul_rn(coef, wwt[i]));
}

// pose <- log(exp(delta) exp(pose)) (:484) with the reference's Pade exponentials, lane-distributed; REF: the logarithm in the
// oracle's closed form (m4_log_ref_f)
template <bool REF = false>
__device__ inline void pose_update_pade_warp(const float (&delta)[6], float rt_pose_e, float (&pose)[6], float* rt_new_e, int lane) {
    const int e = lane & 15;
    const float Ta = se3_exp_pade_warp(delta[0], delta[1], delta[2], delta[3], delta[4], delta[5], e);
    const float Te = m4w_mul(Ta, rt_pose_e, e);
    float T[16];
    ELLC_UNROLL
    for (int i = 0; i < 12; ++i) T[i] = __shfl_sync(kFullWarp, Te, i);
    T[12] = T[13] = T[14] = 0.f; T[15] = 1.f;                  // not read by the logarithm
    if constexpr (REF) m4_log_ref_f(T, pose);
    else m4_log_f(T, pose);
    *rt_new_e = se3_exp_pade_warp(pose[0], pose[1], pose[2], pose[3], pose[4], pose[5], e);
}
// updatePose() given column (lane % 6) of hessianInv in col[0..5]
__device__ inline void update_from_inverse_warp(const float (&col)[6], const float (&b)[6], const float (&weight)[6], float rt_pose_e,
                                                float (&pose)[6], float (&delta)[6], float* weighted_pose, float* rt_new_e, int lane) {
    delta_from_inverse_warp(col, b, weight, delta, weighted_pose, lane);
    pose_update_pade_warp(delta, rt_pose_e, pose, rt_new_e, lane);
}
__device__ inline bool solve_update_warp(const float (&H)[36], const float (&b)[6], const float (&weight)[6], float rt_pose_e,
                                         float (&pose)[6], float (&delta)[6], float* weighted_pose, float* rt_new_e, int lane) {
    float col[6];
    bool ok;
    invert6_lu_warp(H, lane, col, &ok);
    update_from_inverse_warp(col, b, weight, rt_pose_e, pose, delta, weighted_pose, rt_new_e, lane);
    return ok;
}
#endif  // __CUDACC__

}  // namespace ellc
