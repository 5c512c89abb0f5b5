// Geometry stage: DLT triangulation, reprojection error, epipolar correspondence + group ranking.
//
// Replaces, for batches, lib/Helpers.py of the reference:
//   triangulate_point / DLT            :43-84   rows y*P2-P1, P0-x*P2; B = A^T A; singular vector of the smallest
//                                               singular value of B (scipy.linalg.svd) -> X = v[:3]/v[3]
//   calculate_reprojection_error       :102-143 cv.projectPoints(float32(X)) incl. distortion, float32 (u,v),
//                                               mean of squared x/y residuals (px^2)
//   find_point_correspondance_and_object_points :178-280
// B is a symmetric 4x4, so its SVD is its eigen-decomposition: a register-resident cyclic Jacobi solve, one
// point (or candidate group) per thread, FP32 main mode and FP64 check mode (template parameter).  No tensor
// cores: these are tiny independent solves, not dense contractions.
#include "common.cuh"
#include <type_traits>

#define CAM_P 0
#define CAM_R 12
#define CAM_T 21
#define CAM_K 24
#define CAM_D 33

// One MUFU each: the library's rsqrtf / __fdividef wrap the SFU operation into a denormal test and two predicated rescaling
// multiplies when the build does not flush denormals (55 of the 296 instructions of a Jacobi sweep); every argument here is a
// normal number by construction (the tiny terms added below), so the .ftz forms give the same values.
#ifdef MOCAP_EMU
static inline float sfu_rsqrt(float x) { return 1.0f / sqrtf(x); }
static inline float sfu_rcp(float x) { return 1.0f / x; }
#else
__device__ __forceinline__ float sfu_rsqrt(float x) { float y; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float sfu_rcp(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
#endif

// Eigen-decomposition of a symmetric PSD 4x4 (upper triangle b[10]: 00 01 02 03 11 12 13 22 23 33): eigenvalues lam, eigenvectors
// the columns of V.  FP32 main mode: FIVE cyclic sweeps, no data-dependent branch (the lanes of a warp never diverge, nothing is tested
// between rotations).  Five is the budget of the flop count in SURVEY 8d; on the rigs of BASELINE configs 1-5 the smallest eigenvector
// has converged after three to four.
// Rotation from delta = aqq - app: t = 2 apq / (delta + sign(delta) sqrt(delta^2 + 4 apq^2)), c = rsqrt(t^2 + 1), s = t c -- three
// SFU operations (rsqrt, rcp, rsqrt), approximate on purpose: Jacobi rotations are self-correcting, an angle that is off by a few ulp
// leaves a slightly larger off-diagonal for the next sweep.  apq == 0 gives t = 0 (the tiny terms keep 0 / 0 away): identity.
// The vector that comes out carries B's FP32 rounding (about kappa * u, kappa = lam_max / (lam_2 - lam_1)) and what the rotations left:
// over the volume each rig of configs 1-5 sees, X within 7e-7 relative and the reprojection error within 1.3-1.6e-3 px of the FP64
// reference, over the 1e-3 px contract.  dlt_solve takes that back out with one correction step from the rows of A.
__device__ __forceinline__ void jacobi_eig_f32(const float b[10], float lam[4], float V[4][4])
{
    float A[4][4] = {{b[0], b[1], b[2], b[3]}, {b[1], b[4], b[5], b[6]}, {b[2], b[5], b[7], b[8]}, {b[3], b[6], b[8], b[9]}};
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) V[r][c] = r == c ? 1.0f : 0.0f;
#pragma unroll 1
    for (int sweep = 0; sweep < 5; ++sweep) {
#pragma unroll
        for (int p = 0; p < 3; ++p) {
#pragma unroll
            for (int q = p + 1; q < 4; ++q) {
                const float apq = A[p][q];
                const float dl = A[q][q] - A[p][p], two = apq + apq;
                const float ss = dl * dl + two * two;
                const float r = ss * sfu_rsqrt(ss + 1e-37f);
                const float t = two * sfu_rcp(dl + copysignf(r + 1e-30f, dl));
                const float c = sfu_rsqrt(t * t + 1.0f), s = t * c;
                A[p][p] -= t * apq; A[q][q] += t * apq; A[p][q] = 0.0f; A[q][p] = 0.0f;
#pragma unroll
                for (int r2 = 0; r2 < 4; ++r2) {
                    if (r2 != p && r2 != q) {
                        const float arp = A[r2][p], arq = A[r2][q];
                        A[r2][p] = c * arp - s * arq; A[p][r2] = A[r2][p];
                        A[r2][q] = s * arp + c * arq; A[q][r2] = A[r2][q];
                    }
                    const float vrp = V[r2][p], vrq = V[r2][q];
                    V[r2][p] = c * vrp - s * vrq;
                    V[r2][q] = s * vrp + c * vrq;
                }
            }
        }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) lam[k] = A[k][k];
}

// FP64 check mode: IEEE theta / tau rotations, up to twelve cyclic sweeps; the solve ends at a sweep that starts diagonal, and from
// the fourth sweep on an off-diagonal that no longer registers against either diagonal entry is dropped without a rotation (the
// classic Jacobi shortcut), so the last sweeps cost almost nothing.
__device__ __forceinline__ void jacobi_min_eigvec_f64(double b00, double b01, double b02, double b03, double b11, double b12,
                                                      double b13, double b22, double b23, double b33, double v[4])
{
    double A[4][4] = {{b00, b01, b02, b03}, {b01, b11, b12, b13}, {b02, b12, b22, b23}, {b03, b13, b23, b33}};
    double V[4][4] = {{1, 0, 0, 0}, {0, 1, 0, 0}, {0, 0, 1, 0}, {0, 0, 0, 1}};
#pragma unroll 1
    for (int sweep = 0; sweep < 12; ++sweep) {
        const double off = fabs(A[0][1]) + fabs(A[0][2]) + fabs(A[0][3]) + fabs(A[1][2]) + fabs(A[1][3]) + fabs(A[2][3]);
        if (off == 0.0) break;
#pragma unroll
        for (int p = 0; p < 3; ++p) {
#pragma unroll
            for (int q = p + 1; q < 4; ++q) {
                double apq = A[p][q];
                if (sweep >= 3 && apq != 0.0) {
                    const double g = 100.0 * fabs(apq), dp = fabs(A[p][p]), dq = fabs(A[q][q]);
                    if (g + dp == dp && g + dq == dq) { A[p][q] = 0.0; A[q][p] = 0.0; apq = 0.0; }
                }
                if (apq == 0.0) continue;
                const double theta = (A[q][q] - A[p][p]) * (1.0 / (2.0 * apq));
                const double at = fabs(theta);
                double t;
                if (at > 1e15) t = 0.5 * (1.0 / theta);                      // avoid theta^2 overflow
                else { t = 1.0 / (at + sqrt(theta * theta + 1.0)); if (theta < 0.0) t = -t; }
                const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
                const double tau = s * (1.0 / (1.0 + c));
                A[p][p] -= t * apq; A[q][q] += t * apq; A[p][q] = 0.0; A[q][p] = 0.0;
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    if (r != p && r != q) {
                        const double arp = A[r][p], arq = A[r][q];
                        A[r][p] = arp - s * (arq + tau * arp); A[p][r] = A[r][p];
                        A[r][q] = arq + s * (arp - tau * arq); A[q][r] = A[r][q];
                    }
                    const double vrp = V[r][p], vrq = V[r][q];
                    V[r][p] = vrp - s * (vrq + tau * vrp);
                    V[r][q] = vrq + s * (vrp - tau * vrq);
                }
            }
        }
    }
    int k = 0;
    double best = fabs(A[0][0]);
#pragma unroll
    for (int i = 1; i < 4; ++i) { const double e = fabs(A[i][i]); if (e < best) { best = e; k = i; } }
#pragma unroll
    for (int r = 0; r < 4; ++r) v[r] = (k == 0) ? V[r][0] : (k == 1) ? V[r][1] : (k == 2) ? V[r][2] : V[r][3];
}

// twelve consecutive values (a 3x4 P, or R | t of a camera record): three 128-bit loads for floats that are 16-byte aligned
template <typename T> __device__ __forceinline__ void load12(const T* p, T out[12])
{
#pragma unroll
    for (int i = 0; i < 12; ++i) out[i] = p[i];
}
#ifndef MOCAP_EMU
template <> __device__ __forceinline__ void load12<float>(const float* p, float out[12])
{
    if ((((size_t)p) & 15) == 0) {
        const float4 a = ((const float4*)p)[0], b = ((const float4*)p)[1], c = ((const float4*)p)[2];
        out[0] = a.x; out[1] = a.y; out[2] = a.z; out[3] = a.w; out[4] = b.x; out[5] = b.y; out[6] = b.z; out[7] = b.w;
        out[8] = c.x; out[9] = c.y; out[10] = c.z; out[11] = c.w;
    } else {
#pragma unroll
        for (int i = 0; i < 12; ++i) out[i] = p[i];
    }
}
#endif

// The two DLT rows of one view: y*P2 - P1 and P0 - x*P2 (P row-major 3x4)
template <typename T>
__device__ __forceinline__ void dlt_rows(const T Pv[12], T x, T y, T r1[4], T r2[4])
{
#pragma unroll
    for (int c = 0; c < 4; ++c) { r1[c] = y * Pv[8 + c] - Pv[4 + c]; r2[c] = Pv[c] - x * Pv[8 + c]; }
}

// X = v[:3] / v[3] for the smallest eigenvector v of B = A^T A (upper triangle b[10]); views(f) calls f(P, x, y) for each view that
// went into B.  FP32: the Jacobi vector v carries the rounding of B (about kappa * u), so one correction step follows: the residual
// r = sum_i a_i (a_i . v) from the rows of A (not from the rounded B), projected on the other eigenvectors u_k, and
// v -= sum_{k != min} (u_k . r) / (lam_k - lam_min) u_k.  That leaves the rounding of the rows (FP32 P and x, y): every point with
// kappa < 1e3 of tests/test_triangulation_volume.py within 3.2e-7 relative and 4.9e-4 px of the reference on a B200 (CPU emulation build
// 5.3e-7 / 6.2e-4 px).  Plain FP32 dot products a_i . v are enough: Dot2-compensated ones (exact products by fmaf, TwoSum) moved the
// largest error of the emulation build by 2-20 % either way for about 30 more flops per row.
template <class Views>
__device__ __forceinline__ void dlt_solve(const float b[10], Views views, float X[3])
{
    float lam[4], V[4][4];
    jacobi_eig_f32(b, lam, V);
    // column of the smallest |eigenvalue| by selects
    const float e0 = fabsf(lam[0]), e1 = fabsf(lam[1]), e2 = fabsf(lam[2]), e3 = fabsf(lam[3]);
    const bool k01 = e1 < e0, k23 = e3 < e2;
    const float m01 = k01 ? e1 : e0, m23 = k23 ? e3 : e2;
    const bool hi = m23 < m01;
    const float lmin = hi ? (k23 ? lam[3] : lam[2]) : (k01 ? lam[1] : lam[0]);
    float v[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const float a = k01 ? V[r][1] : V[r][0], c = k23 ? V[r][3] : V[r][2];
        v[r] = hi ? c : a;
    }
    // M = sum_{k != min} u_k u_k^T / (lam_k - lam_min) (upper triangle): 10 values live across the view loop instead of V and lam
    float M[10];
#pragma unroll
    for (int i = 0; i < 10; ++i) M[i] = 0.0f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float gap = lam[k] - lmin;
        const float g = gap > 0.0f ? sfu_rcp(gap) : 0.0f;     // 0 for the smallest one itself
        int i = 0;
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int c = r; c < 4; ++c) M[i++] += g * V[r][k] * V[c][k];
    }
    // The rows are formed again rather than kept: an offset the compiler cannot see through stops it from holding every view's P
    // (loaded for B) in registers across the solve, which would double the dense kernels' registers.
    int opaque0 = 0;
    asm volatile("" : "+r"(opaque0));
    float res[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    views([&](const float* P, float x, float y) {
        float Pv[12], r1[4], r2[4];
        load12(P + opaque0, Pv);
        dlt_rows(Pv, x, y, r1, r2);
        const float d1 = r1[0] * v[0] + r1[1] * v[1] + r1[2] * v[2] + r1[3] * v[3];
        const float d2 = r2[0] * v[0] + r2[1] * v[1] + r2[2] * v[2] + r2[3] * v[3];
#pragma unroll
        for (int c = 0; c < 4; ++c) res[c] += r1[c] * d1 + r2[c] * d2;
    });
    const float w[4] = {v[0] - (M[0] * res[0] + M[1] * res[1] + M[2] * res[2] + M[3] * res[3]),
                        v[1] - (M[1] * res[0] + M[4] * res[1] + M[5] * res[2] + M[6] * res[3]),
                        v[2] - (M[2] * res[0] + M[5] * res[1] + M[7] * res[2] + M[8] * res[3]),
                        v[3] - (M[3] * res[0] + M[6] * res[1] + M[8] * res[2] + M[9] * res[3])};
    const float iw = 1.0f / w[3];                          // one IEEE reciprocal instead of three divisions
    X[0] = w[0] * iw; X[1] = w[1] * iw; X[2] = w[2] * iw;
}
template <class Views>
__device__ __forceinline__ void dlt_solve(const double b[10], Views, double X[3])
{
    double v[4];
    jacobi_min_eigvec_f64(b[0], b[1], b[2], b[3], b[4], b[5], b[6], b[7], b[8], b[9], v);
    X[0] = v[0] / v[3]; X[1] = v[1] / v[3]; X[2] = v[2] / v[3];
}

template <typename T>
struct Accum {                          // B = A^T A accumulated view by view
    T b[10];
    __device__ __forceinline__ void clear() {
#pragma unroll
        for (int i = 0; i < 10; ++i) b[i] = (T)0;
    }
    __device__ __forceinline__ void add_row(const T r[4]) {
        b[0] += r[0] * r[0]; b[1] += r[0] * r[1]; b[2] += r[0] * r[2]; b[3] += r[0] * r[3];
        b[4] += r[1] * r[1]; b[5] += r[1] * r[2]; b[6] += r[1] * r[3];
        b[7] += r[2] * r[2]; b[8] += r[2] * r[3]; b[9] += r[3] * r[3];
    }
    __device__ __forceinline__ void add_view(const T* P, T x, T y) {   // P row-major 3x4 (16-byte aligned for T = float)
        T Pv[12];
        load12(P, Pv);
        T r1[4], r2[4];
        dlt_rows(Pv, x, y, r1, r2);
        add_row(r1); add_row(r2);
    }
    // views(f): f(P, x, y) for each view added, in any order (the FP32 solve goes over them once more)
    template <class Views> __device__ __forceinline__ void solve(Views views, T X[3]) { dlt_solve(b, views, X); }
};

// cv.projectPoints restated (SURVEY App. A9).  FP64: reproduces the float32 roundings of X and of (u, v).
template <typename T>
__device__ __forceinline__ void project(const T* cam_pose /*R,t*/, const T* cam_kd /*K,dist*/, const T X[3], T& u, T& v);

template <>
__device__ __forceinline__ void project<double>(const double* pose, const double* kd, const double X[3], double& u, double& v)
{
    double X0 = (double)(float)X[0], X1 = (double)(float)X[1], X2 = (double)(float)X[2];
    const double* R = pose; const double* t = pose + 9;
    // cv::projectPoints: Y = R X + t evaluated left to right, no contraction
    double Yx = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(R[0], X0), __dmul_rn(R[1], X1)), __dmul_rn(R[2], X2)), t[0]);
    double Yy = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(R[3], X0), __dmul_rn(R[4], X1)), __dmul_rn(R[5], X2)), t[1]);
    double Yz = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(R[6], X0), __dmul_rn(R[7], X1)), __dmul_rn(R[8], X2)), t[2]);
    double z = Yz != 0.0 ? __ddiv_rn(1.0, Yz) : 1.0;
    double x = __dmul_rn(Yx, z), y = __dmul_rn(Yy, z);
    double r2 = __dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y));
    double r4 = __dmul_rn(r2, r2), r6 = __dmul_rn(r4, r2);
    double a1 = __dmul_rn(__dmul_rn(2.0, x), y);
    double a2 = __dadd_rn(r2, __dmul_rn(__dmul_rn(2.0, x), x));
    double a3 = __dadd_rn(r2, __dmul_rn(__dmul_rn(2.0, y), y));
    const double* K = kd; const double* d = kd + 9;       // d: k1 k2 p1 p2 k3
    double cdist = __dadd_rn(__dadd_rn(__dadd_rn(1.0, __dmul_rn(d[0], r2)), __dmul_rn(d[1], r4)), __dmul_rn(d[4], r6));
    double xd = __dadd_rn(__dadd_rn(__dmul_rn(x, cdist), __dmul_rn(d[2], a1)), __dmul_rn(d[3], a2));
    double yd = __dadd_rn(__dadd_rn(__dmul_rn(y, cdist), __dmul_rn(d[2], a3)), __dmul_rn(d[3], a1));
    u = (double)(float)__dadd_rn(__dmul_rn(xd, K[0]), K[2]);
    v = (double)(float)__dadd_rn(__dmul_rn(yd, K[4]), K[5]);
}

template <>
__device__ __forceinline__ void project<float>(const float* pose, const float* kd, const float X[3], float& u, float& v)
{
    float Rt[12];
    load12(pose, Rt);
    const float* R = Rt; const float* t = Rt + 9;
    float Yx = R[0] * X[0] + R[1] * X[1] + R[2] * X[2] + t[0];
    float Yy = R[3] * X[0] + R[4] * X[1] + R[5] * X[2] + t[1];
    float Yz = R[6] * X[0] + R[7] * X[1] + R[8] * X[2] + t[2];
    float z = Yz != 0.f ? sfu_rcp(Yz) : 1.f;              // SFU reciprocal (1 ulp): the IEEE division's range test and slow path cost more than the projection's matrix product
    float x = Yx * z, y = Yy * z;
    float r2 = x * x + y * y, r4 = r2 * r2, r6 = r4 * r2;
    float a1 = 2.f * x * y, a2 = r2 + 2.f * x * x, a3 = r2 + 2.f * y * y;
    const float* K = kd; const float* d = kd + 9;
    float cdist = 1.f + d[0] * r2 + d[1] * r4 + d[4] * r6;
    float xd = x * cdist + d[2] * a1 + d[3] * a2;
    float yd = y * cdist + d[2] * a3 + d[3] * a1;
    u = xd * K[0] + K[2];
    v = yd * K[4] + K[5];
}

// camera records in shared memory, converted to T: per camera 38 values (P 12, R 9, t 3, K 9, dist 5)
#define CAM_T_STRIDE 40            // 38 values + padding: P and R | t of every camera start on a 16-byte boundary (floats)
template <typename T>
__device__ __forceinline__ void load_cams(const double* __restrict__ cams, int C, T* sm)
{
    for (int i = threadIdx.x; i < C * CAM_T_STRIDE; i += blockDim.x) {
        int c = i / CAM_T_STRIDE, k = i - c * CAM_T_STRIDE;
        sm[i] = k < 38 ? (T)cams[(size_t)c * MOCAP_CAM_STRIDE + k] : (T)0;
    }
    __syncthreads();
}

// P = K[rank] @ [R|t][cam] (the reference indexes intrinsics by position among the *remaining* views, Helpers.py:58-62)
template <typename T>
__device__ __forceinline__ void make_P(const T* camK, const T* camPose, T* P)
{
    const T* K = camK + CAM_K; const T* R = camPose + CAM_R; const T* t = camPose + CAM_T;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
#pragma unroll
        for (int c = 0; c < 3; ++c) P[4 * r + c] = K[3 * r] * R[c] + K[3 * r + 1] * R[3 + c] + K[3 * r + 2] * R[6 + c];
        P[4 * r + 3] = K[3 * r] * t[0] + K[3 * r + 1] * t[1] + K[3 * r + 2] * t[2];
    }
}

// one image point (x, y): a single 64-bit load for floats (a point list [P][C][2] is 8-byte aligned)
template <typename T> __device__ __forceinline__ void load_xy(const T* p, T& x, T& y) { x = p[0]; y = p[1]; }
#ifndef MOCAP_EMU
template <> __device__ __forceinline__ void load_xy<float>(const float* p, float& x, float& y)
{
    const float2 v = __ldg((const float2*)p);
    x = v.x; y = v.y;
}
#endif

// for (c = 0; c < C; ++c) f(c): unrolled for a compile-time view count CT > 0 (C == CT), else a loop that is not unrolled at all (the
// compiler's partial unrolling of the run-time view loops only adds instructions to the correspondence kernel)
template <int CT, class F>
__device__ __forceinline__ void for_views(int C, F f)
{
    if constexpr (CT > 0) {
#pragma unroll
        for (int c = 0; c < CT; ++c) f(c);
    } else {
#pragma unroll 1
        for (int c = 0; c < C; ++c) f(c);
    }
}

// DLT of one point seen by every view 0 .. C-1: X.  xy(c, x, y) supplies view c's image point.  With sq_residual_all_views (the sum of
// the squared x and y residuals of X over the same views) this is the view loop of every caller whose views are all valid -- the generic
// and the dense triangulation and each candidate group of the correspondence -- so they agree by construction.  The mean (division by
// 2C) stays with the caller: correspondence averages it again over a root's groups.
template <typename T, int CT, class XY>
__device__ __forceinline__ void dlt_all_views(const T* cams, int C, XY xy, T X[3])
{
    auto views = [&](auto f) { for_views<CT>(C, [&](int c) { T x, y; xy(c, x, y); f(cams + c * CAM_T_STRIDE + CAM_P, x, y); }); };
    Accum<T> acc; acc.clear();
    views([&](const T* P, T x, T y) { acc.add_view(P, x, y); });
    acc.solve(views, X);
}

template <typename T, int CT, class XY>
__device__ __forceinline__ T sq_residual_all_views(const T* cams, int C, XY xy, const T X[3])
{
    T s = (T)0;
    for_views<CT>(C, [&](int c) {
        T u, v, x, y;
        project<T>(cams + c * CAM_T_STRIDE + CAM_R, cams + c * CAM_T_STRIDE + CAM_K, X, u, v);
        xy(c, x, y);
        const T dx = x - u, dy = y - v;
        s += dx * dx; s += dy * dy;
    });
    return s;
}

template <typename T, bool TRIANGULATE>
__global__ void __launch_bounds__(128) triangulate_kernel(const T* __restrict__ pts, const uint8_t* __restrict__ valid,
                                                          const T* __restrict__ xyz_in, const double* __restrict__ cams,
                                                          int C, long long n, T* __restrict__ xyz_out, T* __restrict__ err_out)
{
    DYN_SHARED(smraw);
    T* sm = (T*)smraw;
    // blockIdx.y: camera set (mocap_ba_residuals_batch evaluates the same points under several pose hypotheses in one launch)
    cams += (size_t)blockIdx.y * C * MOCAP_CAM_STRIDE;
    if (err_out) err_out += (size_t)blockIdx.y * n;
    if (xyz_out) xyz_out += (size_t)blockIdx.y * n * 3;
    load_cams<T>(cams, C, sm);
    const T nan = (T)NAN;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const T* p = pts + (size_t)i * C * 2;
        const uint8_t* vm = valid ? valid + (size_t)i * C : nullptr;
        T X[3];
        if (TRIANGULATE && !vm && C > 1) {
            auto xy = [&](int c, T& x, T& y) { load_xy(p + 2 * c, x, y); };
            dlt_all_views<T, 0>(sm, C, xy, X);
            if (xyz_out) { xyz_out[(size_t)i * 3] = X[0]; xyz_out[(size_t)i * 3 + 1] = X[1]; xyz_out[(size_t)i * 3 + 2] = X[2]; }
            if (err_out) err_out[i] = sq_residual_all_views<T, 0>(sm, C, xy, X) / (T)(2 * C);
            continue;
        }
        // with a mask, P and the residual take K of the view's rank among the valid views (make_P); given points are reprojected here too
        int nv = 0;
        if (TRIANGULATE) {
            auto views = [&](auto f) {
                int rank = 0;
                for (int c = 0; c < C; ++c) {
                    if (vm && !vm[c]) continue;
                    T x, y, P[12];
                    load_xy(p + 2 * c, x, y);
                    make_P<T>(sm + rank * CAM_T_STRIDE, sm + c * CAM_T_STRIDE, P);
                    f(P, x, y);
                    ++rank;
                }
                return rank;
            };
            Accum<T> acc; acc.clear();
            nv = views([&](const T* P, T x, T y) { acc.add_view(P, x, y); });
            if (nv <= 1) { X[0] = X[1] = X[2] = nan; }
            else acc.solve(views, X);
            if (xyz_out) { xyz_out[(size_t)i * 3] = X[0]; xyz_out[(size_t)i * 3 + 1] = X[1]; xyz_out[(size_t)i * 3 + 2] = X[2]; }
        } else {
            X[0] = xyz_in[(size_t)i * 3]; X[1] = xyz_in[(size_t)i * 3 + 1]; X[2] = xyz_in[(size_t)i * 3 + 2];
            for (int c = 0; c < C; ++c) nv += (!vm || vm[c]);
        }
        if (err_out) {
            T e = nan;
            if (nv > 1) {
                T s = (T)0;
                int rank = 0;
                for (int c = 0; c < C; ++c) {
                    if (vm && !vm[c]) continue;
                    T u, v;
                    project<T>(sm + c * CAM_T_STRIDE + CAM_R, sm + (vm ? rank : c) * CAM_T_STRIDE + CAM_K, X, u, v);
                    T ox, oy;
                    load_xy(p + 2 * c, ox, oy);
                    T dx = ox - u, dy = oy - v;
                    s += dx * dx; s += dy * dy;
                    ++rank;
                }
                e = s / (T)(2 * nv);
            }
            err_out[i] = e;
        }
    }
}

// The bulk case of BASELINE config 5 (every point seen by all CT cameras, FP32): the image points of all CT views loaded into registers
// up front, then the shared view loop unrolled, so the camera records sit at constant shared-memory offsets.
template <int CT>
__global__ void __launch_bounds__(128) triangulate_dense_f32_kernel(const float* __restrict__ pts, const double* __restrict__ cams,
                                                                    long long n, float* __restrict__ xyz_out, float* __restrict__ err_out)
{
    DYN_SHARED(smraw);
    float* sm = (float*)smraw;
    load_cams<float>(cams, CT, sm);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float* p = pts + (size_t)i * CT * 2;
        float px[CT], py[CT];
#pragma unroll
        for (int c = 0; c < CT; ++c) load_xy(p + 2 * c, px[c], py[c]);
        float X[3];
        auto xy = [&](int c, float& x, float& y) { x = px[c]; y = py[c]; };
        dlt_all_views<float, CT>(sm, CT, xy, X);
        if (xyz_out) { xyz_out[(size_t)i * 3] = X[0]; xyz_out[(size_t)i * 3 + 1] = X[1]; xyz_out[(size_t)i * 3 + 2] = X[2]; }
        if (err_out) err_out[i] = sq_residual_all_views<float, CT>(sm, CT, xy, X) / (float)(2 * CT);
    }
}

template <int CT>
static void launch_dense(const void* pts, const double* cams, int64_t n, void* xyz_out, void* err_out, unsigned blocks, cudaStream_t s)
{
    LAUNCH(triangulate_dense_f32_kernel<CT>, blocks, 128, (size_t)CT * CAM_T_STRIDE * sizeof(float), s, (const float*)pts, cams, (long long)n,
           (float*)xyz_out, (float*)err_out);
}

template <typename T>
static int launch_tri(const void* pts, const uint8_t* valid, const void* xyz_in, const double* cams, int C, int64_t n,
                      void* xyz_out, void* err_out, bool tri, cudaStream_t s, int n_sets = 1)
{
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    long long blocks = (n + 127) / 128;
    if (blocks > (long long)sms * 16) blocks = (long long)sms * 16;
    if (blocks < 1) blocks = 1;
    size_t smem = (size_t)C * CAM_T_STRIDE * sizeof(T);
    auto k_tri = triangulate_kernel<T, true>;
    auto k_rep = triangulate_kernel<T, false>;
    const T* no_in = nullptr;
    T* no_out = nullptr;
    if (tri && std::is_same<T, float>::value && !valid && n_sets == 1 && (C == 2 || C == 4 || C == 6 || C == 8 || C == 16)) {
        switch (C) {
        case 2: launch_dense<2>(pts, cams, n, xyz_out, err_out, (unsigned)blocks, s); break;
        case 4: launch_dense<4>(pts, cams, n, xyz_out, err_out, (unsigned)blocks, s); break;
        case 6: launch_dense<6>(pts, cams, n, xyz_out, err_out, (unsigned)blocks, s); break;
        case 8: launch_dense<8>(pts, cams, n, xyz_out, err_out, (unsigned)blocks, s); break;
        default: launch_dense<16>(pts, cams, n, xyz_out, err_out, (unsigned)blocks, s); break;
        }
    } else if (tri) LAUNCH(k_tri, dim3((unsigned)blocks, (unsigned)n_sets), 128, smem, s, (const T*)pts, valid, no_in, cams, C, n, (T*)xyz_out, (T*)err_out);
    else LAUNCH(k_rep, (unsigned)blocks, 128, smem, s, (const T*)pts, valid, (const T*)xyz_in, cams, C, n, no_out, (T*)err_out);
    CUDA_TRY(cudaGetLastError());
    return MOCAP_OK;
}

extern "C" int mocap_triangulate_batch(const void* pts_dev, const uint8_t* valid_dev, const double* cams_dev, int C,
                                       int64_t P, int fp64_mode, void* xyz_out, void* err_out, void* stream)
{
    if (!pts_dev || !cams_dev || !xyz_out || C < 1 || C > MOCAP_MAX_CAMS || P < 0) return MOCAP_ERR_INVALID;
    if (P == 0) return MOCAP_OK;
    if (fp64_mode) return launch_tri<double>(pts_dev, valid_dev, nullptr, cams_dev, C, P, xyz_out, err_out, true, (cudaStream_t)stream);
    return launch_tri<float>(pts_dev, valid_dev, nullptr, cams_dev, C, P, xyz_out, err_out, true, (cudaStream_t)stream);
}

// The residual of bundle_adjustment (lib/Helpers.py:160-167: triangulate_points + calculate_reprojection_errors on all points) for
// n_sets pose hypotheses in ONE launch, FP64 with the reference's roundings: scipy's 2-point finite-difference Jacobian needs the
// residual at x and at x + h e_i for every parameter, i.e. 7 hypotheses per iteration for the 6 parameters of the second camera.
extern "C" int mocap_ba_residuals_batch(const double* pts_dev, const double* cams_sets_dev, int n_sets, int C, int64_t P,
                                        double* err_out, void* stream)
{
    if (!pts_dev || !cams_sets_dev || !err_out || n_sets < 1 || n_sets > 65535 || C < 2 || C > MOCAP_MAX_CAMS || P < 0) return MOCAP_ERR_INVALID;
    if (P == 0) return MOCAP_OK;
    return launch_tri<double>(pts_dev, nullptr, nullptr, cams_sets_dev, C, P, nullptr, err_out, true, (cudaStream_t)stream, n_sets);
}

extern "C" int mocap_reproject_batch(const void* pts_dev, const uint8_t* valid_dev, const void* xyz_dev,
                                     const double* cams_dev, int C, int64_t P, int fp64_mode, void* err_out, void* stream)
{
    if (!pts_dev || !cams_dev || !xyz_dev || !err_out || C < 1 || C > MOCAP_MAX_CAMS || P < 0) return MOCAP_ERR_INVALID;
    if (P == 0) return MOCAP_OK;
    if (fp64_mode) return launch_tri<double>(pts_dev, valid_dev, xyz_dev, cams_dev, C, P, nullptr, err_out, false, (cudaStream_t)stream);
    return launch_tri<float>(pts_dev, valid_dev, xyz_dev, cams_dev, C, P, nullptr, err_out, false, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------------------
// correspondence: CTAs of CORR_RPC roots of one frame-set, then one CTA per frame-set ranks
// ---------------------------------------------------------------------------------------------------------
#define CORR_THREADS 128

// Centroid lists of S frame-sets, camera blocks outermost: xy [C / cpb][S][cpb][max_pts][2], count [C / cpb][S][cpb].  cpb = C is the
// plain [S][C] layout; cpb = cameras per rank is what the shard exchange of the multi-GPU pipeline delivers (one block per source
// rank), so the kernels read the received buffer as it is.  Pt: int32_t (whole-pixel centroids) or float (sub-pixel); both convert to
// float and double exactly, so the epilines, distances, cutoff and ties are the same expressions for either.
template <typename Pt>
struct CorrIn {
    const Pt* xy; const int32_t* count;
    int S, cpb, max_pts;
    __device__ __forceinline__ const Pt* pts(int s, int cam) const {
        const int blk = cam / cpb, ci = cam - blk * cpb;
        return xy + (((size_t)blk * S + s) * cpb + ci) * (size_t)max_pts * 2;
    }
    __device__ __forceinline__ int n(int s, int cam) const {
        const int blk = cam / cpb, ci = cam - blk * cpb;
        return count[((size_t)blk * S + s) * cpb + ci];
    }
};

#ifndef CORR_RPC
#define CORR_RPC 8        // roots per CTA of the candidate / group kernel
#endif
#define CORR_WARPS (CORR_THREADS / 32)

// Workspace of one frame-set: per root the mean error, the first group's point, the first candidate of every camera (the image points
// of the output) and the root's state; per CTA of the group kernel its flags.  Nothing in it grows with max_groups.
struct CorrWs {
    double* rerr; double* rX; int32_t* first; int32_t* vidx; int32_t* flags;
    __device__ __forceinline__ CorrWs(char* wp, int C, int max_pts) {
        rerr = (double*)wp;                                                 // [max_pts] mean error per root
        rX = rerr + max_pts;                                                // [max_pts][3] first group's point
        first = (int32_t*)(rX + 3 * (size_t)max_pts);                       // [max_pts][C] first candidate per camera
        vidx = first + (size_t)max_pts * C;                                 // [max_pts] 0 = complete root, -1 = incomplete
        flags = vidx + max_pts;                                             // [ceil(max_pts / CORR_RPC)] flags per CTA
    }
};

// Part 1, grid (S, ceil(max_pts / CORR_RPC)): candidates per (root, camera), candidate groups, triangulation and mean
// reprojection error of the CTA's roots -> workspace.  Roots are independent until the ranking (Helpers.py:203-273).
template <typename T, typename Pt>
__global__ void __launch_bounds__(CORR_THREADS) correspond_kernel(
    CorrIn<Pt> in, int C, int max_pts,
    const double* __restrict__ Fs, const double* __restrict__ cams, double cutoff, int max_groups,
    int32_t* __restrict__ cand_out, char* __restrict__ ws_base, size_t ws_stride)
{
    DYN_SHARED(smraw);
    T* sm = (T*)smraw;                                                      // camera records [C][CAM_T_STRIDE]
    T* s_cp = sm + C * CAM_T_STRIDE;                                        // candidate points [CORR_RPC][C][MAX_CAND][2] as T
    __shared__ double s_line[CORR_RPC][MOCAP_MAX_CAMS][5];                  // epiline a, b, c, |(a, b)|, far bound per (root, camera)
    __shared__ double s_cd[CORR_RPC][MOCAP_MAX_CAMS][MOCAP_MAX_CAND];       // candidates: distance, point index, count
    __shared__ int s_ck[CORR_RPC][MOCAP_MAX_CAMS][MOCAP_MAX_CAND];
    __shared__ int s_cn[CORR_RPC][MOCAP_MAX_CAMS];
    __shared__ int s_off[CORR_RPC + 1], s_root[CORR_RPC], s_ncomp, s_flags;  // complete roots: group offsets, local root index
    __shared__ T s_part[CORR_RPC][32];                                      // per (complete root, lane of the reference's warp) error sums
    __shared__ T s_e[2][CORR_THREADS];                                      // one round's group errors (double-buffered)
    const int s = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const Pt* root_xy = in.pts(s, 0);
    const int R = min(in.n(s, 0), max_pts);
    const int j0 = blockIdx.y * CORR_RPC, nr = min(CORR_RPC, R - j0);
    if (nr <= 0) return;
    if (tid == 0) s_flags = 0;
    load_cams<T>(cams, C, sm);                                              // ends in __syncthreads
    CorrWs ws(ws_base + (size_t)s * ws_stride, C, max_pts);

    // ---- candidates: one warp per camera, lanes over its points, all roots of the CTA -------------------------------------------
    // Each (root, camera) keeps the MOCAP_MAX_CAND smallest (distance, point index) among the points under the cutoff, merged chunk
    // by chunk of 32 points: a passing point's rank is the number of kept entries at or below its distance (they have smaller
    // indices) plus the passing points of its chunk before it in (distance, index) order.
    int fl = 0;
    for (int i = 1 + wid; i < C; i += CORR_WARPS) {
        if (lane < nr) {                                                    // epiline (FP64 -> f32) of root j0 + lane in camera i
            const int j = j0 + lane;
            const double* F = Fs + (size_t)(i - 1) * 9;
            double x = (double)(float)root_xy[2 * j], y = (double)(float)root_xy[2 * j + 1];
            double a = __dadd_rn(__dadd_rn(__dmul_rn(F[0], x), __dmul_rn(F[1], y)), F[2]);
            double b = __dadd_rn(__dadd_rn(__dmul_rn(F[3], x), __dmul_rn(F[4], y)), F[5]);
            double c = __dadd_rn(__dadd_rn(__dmul_rn(F[6], x), __dmul_rn(F[7], y)), F[8]);
            double nu = __dadd_rn(__dmul_rn(a, a), __dmul_rn(b, b));
            nu = nu != 0.0 ? __ddiv_rn(1.0, sqrt(nu)) : 1.0;
            a = (double)(float)__dmul_rn(a, nu); b = (double)(float)__dmul_rn(b, nu); c = (double)(float)__dmul_rn(c, nu);
            const double den = sqrt(__dadd_rn(__dmul_rn(a, a), __dmul_rn(b, b)));
            double* L = s_line[lane][i];
            L[0] = a; L[1] = b; L[2] = c; L[3] = den;
            // points farther than cutoff + 2e-5 can neither pass the cutoff nor register as a tie: they are rejected on the
            // numerator alone (the margin dwarfs the rounding of the division), so the FP64 divide runs for near points only
            L[4] = __dmul_rn(__dmul_rn(den, cutoff + 2e-5), 1.0 + 1e-12);
            s_cn[lane][i] = 0;
        }
        __syncwarp();
        const Pt* pp = in.pts(s, i);
        const int np = min(in.n(s, i), max_pts);
        for (int k0 = 0; k0 < np; k0 += 32) {
            const int k = k0 + lane;
            double px = 0.0, py = 0.0;
            if (k < np) { px = (double)pp[2 * k]; py = (double)pp[2 * k + 1]; }
#pragma unroll 1
            for (int r = 0; r < nr; ++r) {
                const double* L = s_line[r][i];
                double d = 0.0;
                bool ok = false;
                if (k < np) {
                    const double num = fabs(__dadd_rn(__dadd_rn(__dmul_rn(L[0], px), __dmul_rn(L[1], py)), L[2]));
                    if (!(num > L[4])) {
                        d = __ddiv_rn(num, L[3]);
                        if (fabs(d - cutoff) < 1e-5) fl |= MOCAP_CFLAG_TIE;
                        ok = d < cutoff;
                    }
                }
                const unsigned pass = __ballot_sync(0xffffffffu, ok);
                if (!pass) continue;
                double* cd = s_cd[r][i];
                int* ck = s_ck[r][i];
                const int n = s_cn[r][i];
                const double de = lane < n ? cd[lane] : 0.0;
                const int ke = lane < n ? ck[lane] : 0;
                int below = 0, moved = 0;                                   // passing points before mine / before kept entry `lane`
                for (unsigned m = pass; m; m &= m - 1) {
                    const int q = __ffs(m) - 1;
                    const double dq = __shfl_sync(0xffffffffu, d, q);
                    below += dq < d || (dq == d && q < lane);
                    moved += dq < de;
                }
                for (int e = 0; e < n; ++e) below += cd[e] <= d;
                __syncwarp();
                if (lane < n && lane + moved < MOCAP_MAX_CAND) { cd[lane + moved] = de; ck[lane + moved] = ke; }
                if (ok && below < MOCAP_MAX_CAND) { cd[below] = d; ck[below] = k; }
                const int total = n + __popc(pass);
                if (total > MOCAP_MAX_CAND) fl |= MOCAP_CFLAG_CAND_CAP;
                __syncwarp();
                if (lane == 0) s_cn[r][i] = min(total, MOCAP_MAX_CAND);
                __syncwarp();
            }
        }
    }
    if (fl) atomicOr(&s_flags, fl);
    __syncthreads();

    // ---- stage every candidate point as T, first candidates and cand_out to global ------------------------------------------------
    for (int it = tid; it < nr * C * MOCAP_MAX_CAND; it += CORR_THREADS) {
        const int m = it % MOCAP_MAX_CAND, ri = it / MOCAP_MAX_CAND, r = ri / C, i = ri - r * C, j = j0 + r;
        T* cp = s_cp + (size_t)it * 2;
        if (i == 0) {
            if (m == 0) { cp[0] = (T)root_xy[2 * j]; cp[1] = (T)root_xy[2 * j + 1]; }
            continue;
        }
        const int n = s_cn[r][i], k = m < n ? s_ck[r][i][m] : -1;
        if (k >= 0) { const Pt* pt = in.pts(s, i) + 2 * k; cp[0] = (T)pt[0]; cp[1] = (T)pt[1]; }
        if (m == 0) ws.first[(size_t)j * C + i] = k;
        if (cand_out) cand_out[(((size_t)s * max_pts + j) * C + i) * MOCAP_MAX_CAND + m] = k;
    }
    // complete roots of the CTA and their group counts (the first max_groups groups of each)
    if (wid == 0) {
        long long ng = 1;
        bool complete = C >= 2 && lane < nr;
        if (complete)
            for (int i = 1; i < C; ++i) { int n = s_cn[lane][i]; if (n == 0) complete = false; ng *= n; if (ng > (1LL << 40)) ng = 1LL << 40; }
        if (lane < nr) ws.vidx[j0 + lane] = complete ? 0 : -1;
        if (complete && ng > max_groups) atomicOr(&s_flags, MOCAP_CFLAG_GROUP_CAP);
        const unsigned cm = __ballot_sync(0xffffffffu, complete);
        const int ne = complete ? (int)min(ng, (long long)max_groups) : 0;
        int incl = ne;                                                      // inclusive scan of the group counts over the lanes
        for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
        if (complete) {
            const int q = __popc(cm & ((1u << lane) - 1));
            s_root[q] = lane; s_off[q + 1] = incl;
        }
        if (lane == 0) { s_ncomp = __popc(cm); s_off[0] = 0; }
        if (lane < CORR_RPC) for (int g = 0; g < 32; ++g) s_part[lane][g] = (T)0;
    }
    __syncthreads();

    // ---- candidate groups of all complete roots, CORR_THREADS at a time ---------------------------------------------------------
    // Flat group index f over the complete roots; group g of root q sits at s_off[q] + g.  The mean error keeps the reference
    // kernel's summation order: per root, "lane" g % 32 sums its groups g, g + 32, ... in ascending order from (T)0, then a
    // shuffle tree over offsets 16 .. 1.  Warp 0 adds a round's errors into those 32 partial sums in four steps of 32 consecutive
    // groups (within a step no two groups share a partial sum), so every partial sum takes its groups in ascending order.
    const int ncomp = s_ncomp, total = s_off[ncomp];
    auto root_of = [&](int f) { int q = 0; while (q + 1 < ncomp && f >= s_off[q + 1]) ++q; return q; };
    for (int base = 0, buf = 0; base < total; base += CORR_THREADS, buf ^= 1) {
        const int f = base + tid;
        if (f < total) {
            const int q = root_of(f), r = s_root[q], g = f - s_off[q];
            // mixed radix: camera 1 varies fastest (Helpers.py:239-245 appends the newest camera as the outer loop); 3 bits per view
            unsigned long long dig = 0;
            unsigned rem = (unsigned)g;
            for (int i = 1; i < C; ++i) {
                const unsigned n = (unsigned)s_cn[r][i], qt = rem / n;
                dig |= (unsigned long long)(rem - qt * n) << (3 * i);
                rem = qt;
            }
            const T* cp = s_cp + (size_t)r * C * MOCAP_MAX_CAND * 2;
            auto xy = [&](int i, T& x, T& y) { const T* p = cp + (i * MOCAP_MAX_CAND + (int)((dig >> (3 * i)) & 7)) * 2; x = p[0]; y = p[1]; };
            T X[3];
            dlt_all_views<T, 0>(sm, C, xy, X);
            s_e[buf][tid] = sq_residual_all_views<T, 0>(sm, C, xy, X) / (T)(2 * C);
            if (g == 0) { double* o = ws.rX + 3 * (size_t)(j0 + r); o[0] = (double)X[0]; o[1] = (double)X[1]; o[2] = (double)X[2]; }
        }
        __syncthreads();
        if (wid == 0) {
            for (int w = 0; w < CORR_WARPS; ++w) {
                const int ff = base + w * 32 + lane;
                if (ff < total) { const int q = root_of(ff); s_part[q][(ff - s_off[q]) & 31] += s_e[buf][w * 32 + lane]; }
                __syncwarp();
            }
        }
    }
    __syncthreads();
    for (int q = wid; q < ncomp; q += CORR_WARPS) {
        T esum = s_part[q][lane];
        for (int o = 16; o > 0; o >>= 1) esum += __shfl_down_sync(0xffffffffu, esum, o);     // fixed order: bit-identical on any GPU count
        if (lane == 0) ws.rerr[j0 + s_root[q]] = (double)esum / (double)(s_off[q + 1] - s_off[q]);
    }
    if (tid == 0) ws.flags[blockIdx.y] = s_flags;
}

// Part 2, one CTA per frame-set: the flags of its group CTAs, the complete roots compacted in root order by ballot and prefix sum,
// each ranked by mean error against all others (Helpers.py:274-279), the errors staged in shared memory a tile at a time.
template <typename Pt>
__global__ void __launch_bounds__(CORR_THREADS) correspond_rank_kernel(
    CorrIn<Pt> in, int C, int max_pts, int obj_count,
    double* __restrict__ obj_out, int32_t* __restrict__ n_obj_out, Pt* __restrict__ img_out, int32_t* __restrict__ n_valid_out,
    double* __restrict__ err_out, int32_t* __restrict__ flags_out, char* __restrict__ ws_base, size_t ws_stride)
{
    const int s = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    CorrWs ws(ws_base + (size_t)s * ws_stride, C, max_pts);
    const int R = min(in.n(s, 0), max_pts);
    __shared__ int s_cnt[CORR_WARPS], s_fl[CORR_WARPS];
    __shared__ double s_err[CORR_THREADS];
    __shared__ int s_ok[CORR_THREADS];
    int cnt = 0, fl = 0;
    for (int j = tid; j < R; j += CORR_THREADS) cnt += ws.vidx[j] >= 0;
    for (int b = tid; b < (max(R, 0) + CORR_RPC - 1) / CORR_RPC; b += CORR_THREADS) fl |= ws.flags[b];
    for (int o = 16; o > 0; o >>= 1) { cnt += __shfl_down_sync(0xffffffffu, cnt, o); fl |= __shfl_down_sync(0xffffffffu, fl, o); }
    if (lane == 0) { s_cnt[wid] = cnt; s_fl[wid] = fl; }
    __syncthreads();
    int nvalid = 0;
    fl = 0;
    for (int w = 0; w < CORR_WARPS; ++w) { nvalid += s_cnt[w]; fl |= s_fl[w]; }
    const int n_obj = obj_count > nvalid ? nvalid : min(obj_count + 1, nvalid);
    if (tid == 0) { n_valid_out[s] = nvalid; n_obj_out[s] = n_obj; flags_out[s] = fl; }
    int vbase = 0;                                                          // complete roots before this block of roots
    for (int j0 = 0; j0 < R; j0 += CORR_THREADS) {
        const int j = j0 + tid;
        const bool ok = j < R && ws.vidx[j] >= 0;
        const double e = ok ? ws.rerr[j] : 0.0;
        const unsigned m = __ballot_sync(0xffffffffu, ok);
        __syncthreads();                                                    // s_cnt / s_err of the previous block are consumed
        if (lane == 0) s_cnt[wid] = __popc(m);
        __syncthreads();
        int v = vbase + __popc(m & ((1u << lane) - 1)), nblk = 0;
        for (int w = 0; w < CORR_WARPS; ++w) { const int c = s_cnt[w]; if (w < wid) v += c; nblk += c; }
        vbase += nblk;
        int rank = 0;
        for (int k0 = 0; k0 < R; k0 += CORR_THREADS) {
            __syncthreads();
            const int k = k0 + tid;
            s_ok[tid] = k < R && ws.vidx[k] >= 0;
            s_err[tid] = s_ok[tid] ? ws.rerr[k] : 0.0;
            __syncthreads();
            if (ok)
                for (int t = 0; t < CORR_THREADS; ++t) {
                    const int kk = k0 + t;
                    if (!s_ok[t] || kk == j) continue;
                    const double ek = s_err[t];
                    rank += (ek < e) || (ek == e && kk < j);
                }
        }
        if (!ok) continue;
        if (rank < n_obj) {
            double* o = obj_out + ((size_t)s * max_pts + rank) * 3;
            o[0] = ws.rX[3 * j]; o[1] = ws.rX[3 * j + 1]; o[2] = ws.rX[3 * j + 2];
        }
        err_out[(size_t)s * max_pts + v] = e;
        Pt* io = img_out + ((size_t)s * max_pts + v) * C * 2;
        for (int i = 0; i < C; ++i) {
            const int k = i == 0 ? j : ws.first[(size_t)j * C + i];
            const Pt* pt = in.pts(s, i) + 2 * k;
            io[2 * i] = pt[0];
            io[2 * i + 1] = pt[1];
        }
    }
}

static size_t corr_ws_stride(int C, int max_pts)
{
    size_t b = (size_t)max_pts * 4 * 8 + ((size_t)max_pts * C + (size_t)max_pts + (size_t)cdiv(max_pts, CORR_RPC)) * 4;
    return (b + 255) & ~(size_t)255;
}

extern "C" size_t mocap_correspond_workspace_bytes(int S, int C, int max_pts, int max_groups)
{
    (void)max_groups;
    if (S <= 0 || C <= 0 || max_pts <= 0) return 0;
    return corr_ws_stride(C, max_pts) * (size_t)S;
}

// every correspondence entry point: int32 (Pt = int32_t) or float32 (Pt = float) centroid lists, camera-blocked
template <typename Pt>
static int correspond_blocked(const Pt* xy_dev, const int32_t* count_dev, int S, int C, int max_pts, int cams_per_block,
                              const double* F_dev, const double* cams_dev, double cutoff, int obj_count,
                              int max_groups, int fp64_mode,
                              double* obj_out, int32_t* n_obj_out, Pt* img_out, int32_t* n_valid_out,
                              double* err_out, int32_t* cand_out, int32_t* flags_out,
                              void* workspace, size_t workspace_bytes, void* stream)
{
    if (cams_per_block < 1 || (C > 0 && C % cams_per_block != 0)) return MOCAP_ERR_INVALID;
    if (!xy_dev || !count_dev || !cams_dev || !obj_out || !n_obj_out || !img_out || !n_valid_out || !err_out || !flags_out || !workspace)
        return MOCAP_ERR_INVALID;
    if (S < 0 || C < 1 || C > MOCAP_MAX_CAMS || max_pts < 1 || max_groups < 1 || obj_count < 0) return MOCAP_ERR_INVALID;
    if (C > 1 && !F_dev) return MOCAP_ERR_INVALID;
    if (S == 0) return MOCAP_OK;
    size_t stride = corr_ws_stride(C, max_pts);
    if (workspace_bytes < stride * (size_t)S) return MOCAP_ERR_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    dim3 grid(S, cdiv(max_pts, CORR_RPC));
    CorrIn<Pt> in;
    in.xy = xy_dev; in.count = count_dev; in.S = S; in.cpb = cams_per_block; in.max_pts = max_pts;
    auto corr_f64 = correspond_kernel<double, Pt>;
    auto corr_f32 = correspond_kernel<float, Pt>;
    auto rank = correspond_rank_kernel<Pt>;
    const size_t smem_per_T = (size_t)C * (CAM_T_STRIDE + CORR_RPC * MOCAP_MAX_CAND * 2);
    if (fp64_mode)
        LAUNCH(corr_f64, grid, CORR_THREADS, smem_per_T * sizeof(double), s,
            in, C, max_pts, F_dev, cams_dev, cutoff, max_groups, cand_out, (char*)workspace, stride);
    else
        LAUNCH(corr_f32, grid, CORR_THREADS, smem_per_T * sizeof(float), s,
            in, C, max_pts, F_dev, cams_dev, cutoff, max_groups, cand_out, (char*)workspace, stride);
    LAUNCH(rank, S, CORR_THREADS, 0, s, in, C, max_pts, obj_count, obj_out, n_obj_out, img_out,
           n_valid_out, err_out, flags_out, (char*)workspace, stride);
    CUDA_TRY(cudaGetLastError());
    return MOCAP_OK;
}

extern "C" int mocap_correspond_batch_blocked(const int32_t* xy_dev, const int32_t* count_dev, int S, int C, int max_pts, int cams_per_block,
                                              const double* F_dev, const double* cams_dev, double cutoff, int obj_count,
                                              int max_groups, int fp64_mode,
                                              double* obj_out, int32_t* n_obj_out, int32_t* img_out, int32_t* n_valid_out,
                                              double* err_out, int32_t* cand_out, int32_t* flags_out,
                                              void* workspace, size_t workspace_bytes, void* stream)
{
    return correspond_blocked(xy_dev, count_dev, S, C, max_pts, cams_per_block, F_dev, cams_dev, cutoff, obj_count, max_groups, fp64_mode,
                              obj_out, n_obj_out, img_out, n_valid_out, err_out, cand_out, flags_out, workspace, workspace_bytes, stream);
}

extern "C" int mocap_correspond_batch_subpixel(const float* xy_dev, const int32_t* count_dev, int S, int C, int max_pts, int cams_per_block,
                                               const double* F_dev, const double* cams_dev, double cutoff, int obj_count,
                                               int max_groups, int fp64_mode,
                                               double* obj_out, int32_t* n_obj_out, float* img_out, int32_t* n_valid_out,
                                               double* err_out, int32_t* cand_out, int32_t* flags_out,
                                               void* workspace, size_t workspace_bytes, void* stream)
{
    return correspond_blocked(xy_dev, count_dev, S, C, max_pts, cams_per_block, F_dev, cams_dev, cutoff, obj_count, max_groups, fp64_mode,
                              obj_out, n_obj_out, img_out, n_valid_out, err_out, cand_out, flags_out, workspace, workspace_bytes, stream);
}

extern "C" int mocap_correspond_batch(const int32_t* xy_dev, const int32_t* count_dev, int S, int C, int max_pts,
                                      const double* F_dev, const double* cams_dev, double cutoff, int obj_count,
                                      int max_groups, int fp64_mode,
                                      double* obj_out, int32_t* n_obj_out, int32_t* img_out, int32_t* n_valid_out,
                                      double* err_out, int32_t* cand_out, int32_t* flags_out,
                                      void* workspace, size_t workspace_bytes, void* stream)
{
    return correspond_blocked(xy_dev, count_dev, S, C, max_pts, C, F_dev, cams_dev, cutoff, obj_count, max_groups, fp64_mode,
                              obj_out, n_obj_out, img_out, n_valid_out, err_out, cand_out, flags_out, workspace, workspace_bytes, stream);
}
