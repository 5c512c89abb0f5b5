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

template <typename T> struct Num;
template <> struct Num<float> {
    static __device__ __forceinline__ float sqrt_(float x) { return sqrtf(x); }
    static __device__ __forceinline__ float abs_(float x) { return fabsf(x); }
    static __device__ __forceinline__ float tiny() { return 1e-30f; }
    // Jacobi rotations are self-correcting: an angle that is off by a few ulp only leaves a slightly larger off-diagonal
    // for the next sweep, so the FP32 main mode uses the SFU reciprocal / rsqrt (the FP64 check mode stays IEEE)
    static __device__ __forceinline__ float rcp_(float x) { return __frcp_rn(x); }
    static __device__ __forceinline__ float rsqrt_(float x) { return rsqrtf(x); }
    static constexpr int sweeps = 8;
};
template <> struct Num<double> {
    static __device__ __forceinline__ double sqrt_(double x) { return sqrt(x); }
    static __device__ __forceinline__ double abs_(double x) { return fabs(x); }
    static __device__ __forceinline__ double tiny() { return 1e-280; }
    static __device__ __forceinline__ double rcp_(double x) { return 1.0 / x; }
    static __device__ __forceinline__ double rsqrt_(double x) { return 1.0 / sqrt(x); }
    static constexpr int sweeps = 12;
};

// Smallest-eigenvalue eigenvector of a symmetric PSD 4x4 (upper triangle a[10]: 00 01 02 03 11 12 13 22 23 33).
// FP32 main mode: FIVE cyclic sweeps, no data-dependent branch (the lanes of a warp never diverge, nothing is tested between
// rotations).  Five is the budget of the flop count in SURVEY 8d; on the rigs of BASELINE configs 1-5 the smallest eigenvector has
// converged to FP32 round-off after three to four (max relative error of X against the FP64 SVD 7e-7 at every count >= 4).
// Rotation from delta = aqq - app: t = 2 apq / (delta + sign(delta) sqrt(delta^2 + 4 apq^2)), c = rsqrt(t^2 + 1), s = t c -- three
// SFU operations (rsqrt, rcp, rsqrt), approximate on purpose: Jacobi rotations are self-correcting, an angle that is off by a few ulp
// leaves a slightly larger off-diagonal for the next sweep.  apq == 0 gives t = 0 (the tiny terms keep 0 / 0 away): identity.
__device__ __forceinline__ void jacobi_min_eigvec_f32(float b00, float b01, float b02, float b03, float b11, float b12, float b13,
                                                      float b22, float b23, float b33, float v[4])
{
    float A[4][4] = {{b00, b01, b02, b03}, {b01, b11, b12, b13}, {b02, b12, b22, b23}, {b03, b13, b23, b33}};
    float V[4][4] = {{1, 0, 0, 0}, {0, 1, 0, 0}, {0, 0, 1, 0}, {0, 0, 0, 1}};
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
    // column of the smallest |eigenvalue| by selects
    const float e0 = fabsf(A[0][0]), e1 = fabsf(A[1][1]), e2 = fabsf(A[2][2]), e3 = fabsf(A[3][3]);
    const bool k01 = e1 < e0, k23 = e3 < e2;
    const float m01 = k01 ? e1 : e0, m23 = k23 ? e3 : e2;
    const bool hi = m23 < m01;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const float a = k01 ? V[r][1] : V[r][0], b = k23 ? V[r][3] : V[r][2];
        v[r] = hi ? b : a;
    }
}

template <typename T>
__device__ __forceinline__ void jacobi_min_eigvec(T b00, T b01, T b02, T b03, T b11, T b12, T b13, T b22, T b23, T b33, T v[4])
{
    T A[4][4] = {{b00, b01, b02, b03}, {b01, b11, b12, b13}, {b02, b12, b22, b23}, {b03, b13, b23, b33}};
    T V[4][4] = {{1, 0, 0, 0}, {0, 1, 0, 0}, {0, 0, 1, 0}, {0, 0, 0, 1}};
#pragma unroll 1
    for (int sweep = 0; sweep < Num<T>::sweeps; ++sweep) {
        T off = Num<T>::abs_(A[0][1]) + Num<T>::abs_(A[0][2]) + Num<T>::abs_(A[0][3]) +
                Num<T>::abs_(A[1][2]) + Num<T>::abs_(A[1][3]) + Num<T>::abs_(A[2][3]);
        if (off == (T)0) break;
#pragma unroll
        for (int p = 0; p < 3; ++p) {
#pragma unroll
            for (int q = p + 1; q < 4; ++q) {
                T apq = A[p][q];
                // after the first sweeps an off-diagonal that no longer registers against either diagonal entry is dropped
                // without a rotation (the classic Jacobi shortcut), so the last sweeps cost almost nothing
                if (sweep >= 3 && apq != (T)0) {
                    T g = (T)100 * Num<T>::abs_(apq), dp = Num<T>::abs_(A[p][p]), dq = Num<T>::abs_(A[q][q]);
                    if (g + dp == dp && g + dq == dq) { A[p][q] = (T)0; A[q][p] = (T)0; apq = (T)0; }
                }
                if (sizeof(T) == 4 && apq != (T)0) {
                    // FP32 main mode: the rotation from delta = aqq - app directly, t = 2 apq / (delta + sign(delta) sqrt(delta^2 +
                    // 4 apq^2)), applied as (c, s) -- three SFU operations (sqrt, rcp, rsqrt) instead of the five of the theta /
                    // tau form below, which the FP64 check mode keeps
                    T dl = A[q][q] - A[p][p], two = (T)2 * apq;
                    T r = Num<T>::sqrt_(dl * dl + two * two);
                    T t = two * Num<T>::rcp_(dl + (dl < (T)0 ? -r : r));
                    T c = Num<T>::rsqrt_(t * t + (T)1), s = t * c;
                    A[p][p] -= t * apq; A[q][q] += t * apq; A[p][q] = (T)0; A[q][p] = (T)0;
#pragma unroll
                    for (int r2 = 0; r2 < 4; ++r2) {
                        if (r2 != p && r2 != q) {
                            T arp = A[r2][p], arq = A[r2][q];
                            A[r2][p] = c * arp - s * arq; A[p][r2] = A[r2][p];
                            A[r2][q] = s * arp + c * arq; A[q][r2] = A[r2][q];
                        }
                        T vrp = V[r2][p], vrq = V[r2][q];
                        V[r2][p] = c * vrp - s * vrq;
                        V[r2][q] = s * vrp + c * vrq;
                    }
                } else if (apq != (T)0) {
                    T theta = (A[q][q] - A[p][p]) * Num<T>::rcp_((T)2 * apq);
                    T at = Num<T>::abs_(theta);
                    T t;
                    if (at > (T)1e15) t = (T)0.5 * Num<T>::rcp_(theta);         // avoid theta^2 overflow
                    else { t = Num<T>::rcp_(at + Num<T>::sqrt_(theta * theta + (T)1)); if (theta < (T)0) t = -t; }
                    T c = Num<T>::rsqrt_(t * t + (T)1), s = t * c;
                    T tau = s * Num<T>::rcp_((T)1 + c);
                    A[p][p] -= t * apq; A[q][q] += t * apq; A[p][q] = (T)0; A[q][p] = (T)0;
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        if (r != p && r != q) {
                            T arp = A[r][p], arq = A[r][q];
                            A[r][p] = arp - s * (arq + tau * arp); A[p][r] = A[r][p];
                            A[r][q] = arq + s * (arp - tau * arq); A[q][r] = A[r][q];
                        }
                        T vrp = V[r][p], vrq = V[r][q];
                        V[r][p] = vrp - s * (vrq + tau * vrp);
                        V[r][q] = vrq + s * (vrp - tau * vrq);
                    }
                }
            }
        }
    }
    int k = 0;
    T best = Num<T>::abs_(A[0][0]);
#pragma unroll
    for (int i = 1; i < 4; ++i) { T e = Num<T>::abs_(A[i][i]); if (e < best) { best = e; k = i; } }
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
#pragma unroll
        for (int c = 0; c < 4; ++c) { r1[c] = y * Pv[8 + c] - Pv[4 + c]; r2[c] = Pv[c] - x * Pv[8 + c]; }
        add_row(r1); add_row(r2);
    }
    __device__ __forceinline__ void solve(T X[3]) {
        T v[4];
        if (sizeof(T) == 4) {
            float w[4];
            jacobi_min_eigvec_f32((float)b[0], (float)b[1], (float)b[2], (float)b[3], (float)b[4], (float)b[5], (float)b[6], (float)b[7],
                                  (float)b[8], (float)b[9], w);
            const float iw = 1.0f / w[3];                      // one IEEE reciprocal instead of three divisions
            X[0] = (T)(w[0] * iw); X[1] = (T)(w[1] * iw); X[2] = (T)(w[2] * iw);
            return;
        }
        jacobi_min_eigvec<T>(b[0], b[1], b[2], b[3], b[4], b[5], b[6], b[7], b[8], b[9], v);
        X[0] = v[0] / v[3]; X[1] = v[1] / v[3]; X[2] = v[2] / v[3];
    }
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
        int nv = 0;
        if (TRIANGULATE) {
            Accum<T> acc; acc.clear();
            for (int c = 0; c < C; ++c) {
                if (vm && !vm[c]) continue;
                T x, y;
                load_xy(p + 2 * c, x, y);
                if (vm) { T P[12]; make_P<T>(sm + nv * CAM_T_STRIDE, sm + c * CAM_T_STRIDE, P); acc.add_view(P, x, y); }
                else acc.add_view(sm + c * CAM_T_STRIDE + CAM_P, x, y);
                ++nv;
            }
            if (nv <= 1) { X[0] = X[1] = X[2] = nan; }
            else acc.solve(X);
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

// The bulk case of BASELINE config 5 (every point seen by all CT cameras, FP32, triangulation + reprojection error): the same
// arithmetic as triangulate_kernel<float, true> with the view loops unrolled -- the camera records sit at constant shared-memory
// offsets, no validity tests, no per-view address arithmetic (in the generic kernel ~45 of the ~150 instructions per view).
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
        Accum<float> acc; acc.clear();
#pragma unroll
        for (int c = 0; c < CT; ++c) acc.add_view(sm + c * CAM_T_STRIDE + CAM_P, px[c], py[c]);
        float X[3];
        acc.solve(X);
        if (xyz_out) { xyz_out[(size_t)i * 3] = X[0]; xyz_out[(size_t)i * 3 + 1] = X[1]; xyz_out[(size_t)i * 3 + 2] = X[2]; }
        if (err_out) {
            float s = 0.f;
#pragma unroll
            for (int c = 0; c < CT; ++c) {
                float u, v;
                project<float>(sm + c * CAM_T_STRIDE + CAM_R, sm + c * CAM_T_STRIDE + CAM_K, X, u, v);
                const float dx = px[c] - u, dy = py[c] - v;
                s += dx * dx; s += dy * dy;
            }
            err_out[i] = s / (float)(2 * CT);
        }
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
    if (tri && sizeof(T) == 4 && !valid && n_sets == 1 && (C == 2 || C == 4 || C == 6 || C == 8 || C == 16)) {
        if (C == 2) launch_dense<2>(pts, cams, n, xyz_out, err_out, (unsigned)blocks, s);
        else if (C == 4) launch_dense<4>(pts, cams, n, xyz_out, err_out, (unsigned)blocks, s);
        else if (C == 6) launch_dense<6>(pts, cams, n, xyz_out, err_out, (unsigned)blocks, s);
        else if (C == 8) launch_dense<8>(pts, cams, n, xyz_out, err_out, (unsigned)blocks, s);
        else launch_dense<16>(pts, cams, n, xyz_out, err_out, (unsigned)blocks, s);
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
// correspondence: one CTA per frame-set
// ---------------------------------------------------------------------------------------------------------
#define CORR_THREADS 128

struct CorrWs { int32_t* cand; int32_t* ncand; };

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

// Part 1, grid (S, ceil(max_pts / CORR_RPC)): candidates per (root, camera), candidate groups, triangulation and mean
// reprojection error of the CTA's roots -> workspace.  Roots are independent until the ranking (Helpers.py:203-273).
template <typename T, typename Pt>
__global__ void __launch_bounds__(CORR_THREADS) correspond_kernel(
    CorrIn<Pt> in, int C, int max_pts,
    const double* __restrict__ Fs, const double* __restrict__ cams, double cutoff, int max_groups,
    int32_t* __restrict__ cand_out, int32_t* __restrict__ flags_out, char* __restrict__ ws_base, size_t ws_stride)
{
    DYN_SHARED(smraw);
    T* sm = (T*)smraw;
    const int s = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nw = blockDim.x >> 5;
    const Pt* root_xy = in.pts(s, 0);
    const int R = min(in.n(s, 0), max_pts);
    const int j0 = blockIdx.y * CORR_RPC, j1 = min(j0 + CORR_RPC, R);
    if (j0 >= R) return;
    load_cams<T>(cams, C, sm);
    __shared__ int s_flags;
    if (tid == 0) s_flags = 0;
    char* wp = ws_base + (size_t)s * ws_stride;
    double* rerr = (double*)wp;                                             // [max_pts] mean error per root
    double* rX = rerr + max_pts;                                            // [max_pts][3] first group's point
    int32_t* cand = (int32_t*)(rX + 3 * (size_t)max_pts);                   // [max_pts][C][MAX_CAND]
    int32_t* ncand = cand + (size_t)max_pts * C * MOCAP_MAX_CAND;           // [max_pts][C]
    int32_t* vidx = ncand + (size_t)max_pts * C;                            // [max_pts] 0 = complete root, -1 = incomplete
    __syncthreads();

    // ---- candidates per (root, camera): epiline (FP64 -> f32) and point-line distances (FP64) --------------------------
    for (int it = tid; it < (j1 - j0) * C; it += blockDim.x) {
        int j = j0 + it / C, i = it % C;
        int32_t* cl = cand + ((size_t)j * C + i) * MOCAP_MAX_CAND;
        if (i == 0) { ncand[j * C] = 1; cl[0] = j; continue; }
        const double* F = Fs + (size_t)(i - 1) * 9;
        double x = (double)(float)root_xy[2 * j], y = (double)(float)root_xy[2 * j + 1];      // root is camera-0 point j
        double a = __dadd_rn(__dadd_rn(__dmul_rn(F[0], x), __dmul_rn(F[1], y)), F[2]);
        double b = __dadd_rn(__dadd_rn(__dmul_rn(F[3], x), __dmul_rn(F[4], y)), F[5]);
        double c = __dadd_rn(__dadd_rn(__dmul_rn(F[6], x), __dmul_rn(F[7], y)), F[8]);
        double nu = __dadd_rn(__dmul_rn(a, a), __dmul_rn(b, b));
        nu = nu != 0.0 ? __ddiv_rn(1.0, sqrt(nu)) : 1.0;
        a = (double)(float)__dmul_rn(a, nu); b = (double)(float)__dmul_rn(b, nu); c = (double)(float)__dmul_rn(c, nu);
        double den = sqrt(__dadd_rn(__dmul_rn(a, a), __dmul_rn(b, b)));
        const Pt* pp = in.pts(s, i);
        int np = min(in.n(s, i), max_pts), n = 0, fl = 0;
        double dist[MOCAP_MAX_CAND];
        // points farther than cutoff + 2e-5 can neither pass the cutoff nor register as a tie: they are rejected on the
        // numerator alone (the margin dwarfs the rounding of the division), so the FP64 divide runs for near points only
        const double far = __dmul_rn(__dmul_rn(den, cutoff + 2e-5), 1.0 + 1e-12);
        for (int k = 0; k < np; ++k) {
            double num = fabs(__dadd_rn(__dadd_rn(__dmul_rn(a, (double)pp[2 * k]), __dmul_rn(b, (double)pp[2 * k + 1])), c));
            if (num > far) continue;
            double d = __ddiv_rn(num, den);
            if (fabs(d - cutoff) < 1e-5) fl |= MOCAP_CFLAG_TIE;
            if (!(d < cutoff)) continue;
            int pos;                                           // keep the MOCAP_MAX_CAND smallest, stable on ties
            if (n < MOCAP_MAX_CAND) { pos = n; ++n; }
            else { fl |= MOCAP_CFLAG_CAND_CAP; if (!(d < dist[MOCAP_MAX_CAND - 1])) continue; pos = MOCAP_MAX_CAND - 1; }
            while (pos > 0 && d < dist[pos - 1]) { dist[pos] = dist[pos - 1]; cl[pos] = cl[pos - 1]; --pos; }
            dist[pos] = d; cl[pos] = k;
        }
        ncand[j * C + i] = n;
        if (fl) atomicOr(&s_flags, fl);
        if (cand_out) {
            int32_t* co = cand_out + (((size_t)s * max_pts + j) * C + i) * MOCAP_MAX_CAND;
            for (int k = 0; k < MOCAP_MAX_CAND; ++k) co[k] = k < n ? cl[k] : -1;
        }
    }
    __syncthreads();

    // ---- per root (one warp each): enumerate candidate groups, triangulate, mean reprojection error ----------------------
    for (int j = j0 + wid; j < j1; j += nw) {
        long long ng = 1;
        bool complete = C >= 2;
        for (int i = 1; i < C; ++i) { int n = ncand[j * C + i]; if (n == 0) complete = false; ng *= n; if (ng > (1LL << 40)) ng = 1LL << 40; }
        if (!complete) { if (lane == 0) vidx[j] = -1; continue; }
        int ne = (int)min(ng, (long long)max_groups);
        if (ng > max_groups && lane == 0) atomicOr(&s_flags, MOCAP_CFLAG_GROUP_CAP);
        T esum = (T)0;
        T X0[3] = {0, 0, 0};
        for (int g = lane; g < ne; g += 32) {
            // mixed radix: camera 1 varies fastest (Helpers.py:239-245 appends the newest camera as the outer loop)
            Accum<T> acc; acc.clear();
            T px[MOCAP_MAX_CAMS], py[MOCAP_MAX_CAMS];
            int rem = g;
            for (int i = 0; i < C; ++i) {
                int k;
                if (i == 0) k = j;
                else { int n = ncand[j * C + i]; int q = rem / n; k = cand[((size_t)j * C + i) * MOCAP_MAX_CAND + (rem - q * n)]; rem = q; }
                const Pt* pt = in.pts(s, i) + 2 * k;
                px[i] = (T)pt[0]; py[i] = (T)pt[1];
                acc.add_view(sm + i * CAM_T_STRIDE + CAM_P, px[i], py[i]);
            }
            T X[3];
            acc.solve(X);
            T sq = (T)0;
            for (int i = 0; i < C; ++i) {
                T u, v;
                project<T>(sm + i * CAM_T_STRIDE + CAM_R, sm + i * CAM_T_STRIDE + CAM_K, X, u, v);
                T dx = px[i] - u, dy = py[i] - v;
                sq += dx * dx; sq += dy * dy;
            }
            esum += sq / (T)(2 * C);
            if (g == 0) { X0[0] = X[0]; X0[1] = X[1]; X0[2] = X[2]; }
        }
        // fixed-order warp reduction (bit-identical on any GPU count)
        for (int o = 16; o > 0; o >>= 1) esum += __shfl_down_sync(0xffffffffu, esum, o);
        if (lane == 0) {
            rerr[j] = (double)esum / (double)ne;
            rX[3 * j] = (double)X0[0]; rX[3 * j + 1] = (double)X0[1]; rX[3 * j + 2] = (double)X0[2];
            vidx[j] = 0;
        }
    }
    __syncthreads();
    if (tid == 0 && s_flags) atomicOr(&flags_out[s], s_flags);
}

// Part 2, one CTA per frame-set: compact the complete roots in root order, rank them by mean error (Helpers.py:274-279)
template <typename Pt>
__global__ void __launch_bounds__(CORR_THREADS) correspond_rank_kernel(
    CorrIn<Pt> in, int C, int max_pts, int obj_count,
    double* __restrict__ obj_out, int32_t* __restrict__ n_obj_out, Pt* __restrict__ img_out, int32_t* __restrict__ n_valid_out,
    double* __restrict__ err_out, char* __restrict__ ws_base, size_t ws_stride)
{
    const int s = blockIdx.x, tid = threadIdx.x;
    char* wp = ws_base + (size_t)s * ws_stride;
    double* rerr = (double*)wp;
    double* rX = rerr + max_pts;
    int32_t* cand = (int32_t*)(rX + 3 * (size_t)max_pts);
    int32_t* ncand = cand + (size_t)max_pts * C * MOCAP_MAX_CAND;
    int32_t* vidx = ncand + (size_t)max_pts * C;
    const int R = min(in.n(s, 0), max_pts);
    __shared__ int s_nvalid;
    if (tid == 0) {
        int n = 0;
        for (int j = 0; j < R; ++j) if (vidx[j] >= 0) vidx[j] = n++;
        s_nvalid = n;
    }
    __syncthreads();
    const int nvalid = s_nvalid;
    for (int j = tid; j < R; j += blockDim.x) {
        int v = vidx[j];
        if (v < 0) continue;
        double e = rerr[j];
        int rank = 0;
        for (int k = 0; k < R; ++k) {
            if (vidx[k] < 0 || k == j) continue;
            double ek = rerr[k];
            rank += (ek < e) || (ek == e && k < j);
        }
        int n_obj = obj_count > nvalid ? nvalid : min(obj_count + 1, nvalid);
        if (rank < n_obj) {
            double* o = obj_out + ((size_t)s * max_pts + rank) * 3;
            o[0] = rX[3 * j]; o[1] = rX[3 * j + 1]; o[2] = rX[3 * j + 2];
        }
        err_out[(size_t)s * max_pts + v] = e;
        Pt* io = img_out + ((size_t)s * max_pts + v) * C * 2;
        for (int i = 0; i < C; ++i) {
            int k = i == 0 ? j : cand[((size_t)j * C + i) * MOCAP_MAX_CAND];
            const Pt* pt = in.pts(s, i) + 2 * k;
            io[2 * i] = pt[0];
            io[2 * i + 1] = pt[1];
        }
    }
    if (tid == 0) {
        n_valid_out[s] = nvalid;
        n_obj_out[s] = obj_count > nvalid ? nvalid : min(obj_count + 1, nvalid);
    }
}

static size_t corr_ws_stride(int C, int max_pts)
{
    size_t b = ((size_t)max_pts * C * MOCAP_MAX_CAND + (size_t)max_pts * C + (size_t)max_pts) * 4 + (size_t)max_pts * 4 * 8;
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
    CUDA_TRY(cudaMemsetAsync(flags_out, 0, (size_t)S * 4, s));
    dim3 grid(S, cdiv(max_pts, CORR_RPC));
    CorrIn<Pt> in;
    in.xy = xy_dev; in.count = count_dev; in.S = S; in.cpb = cams_per_block; in.max_pts = max_pts;
    auto corr_f64 = correspond_kernel<double, Pt>;
    auto corr_f32 = correspond_kernel<float, Pt>;
    auto rank = correspond_rank_kernel<Pt>;
    if (fp64_mode)
        LAUNCH(corr_f64, grid, CORR_THREADS, (size_t)C * CAM_T_STRIDE * sizeof(double), s,
            in, C, max_pts, F_dev, cams_dev, cutoff, max_groups, cand_out, flags_out, (char*)workspace, stride);
    else
        LAUNCH(corr_f32, grid, CORR_THREADS, (size_t)C * CAM_T_STRIDE * sizeof(float), s,
            in, C, max_pts, F_dev, cams_dev, cutoff, max_groups, cand_out, flags_out, (char*)workspace, stride);
    LAUNCH(rank, S, CORR_THREADS, 0, s, in, C, max_pts, obj_count, obj_out, n_obj_out, img_out,
           n_valid_out, err_out, (char*)workspace, stride);
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
