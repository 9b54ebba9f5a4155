// deskew.cuh — ImageProjection::projectPointCloud + deskewPoint + findRotation on the GPU
// (src/imageProjection.cpp:568-598, 536-566, 493-518).  liorf keeps no range image: the function is
// filter → per-point IMU-rotation deskew → ORDER-PRESERVING append.  Bandwidth-bound streaming:
// 24 B in per raw point, 16 B out per kept point.
//
//   k_first_kept : finds the first point that survives the filters (it fixes transStartInverse, :549-553)
//   scan kernel  : keep flag → exclusive scan (decoupled look-back) → deskew + ordered store
#pragma once
#include "prims.cuh"

namespace liorf {

struct RawPoint { float x, y, z, intensity; unsigned short ring, pad; float time; };   // VelodynePointXYZIRT payload (:4-15)
static_assert(sizeof(RawPoint) == 24, "raw point must be 24 bytes");

struct DeskewParams { float lidarMinRange, lidarMaxRange; int N_SCAN, downsampleRate, point_filter_num; };

struct ImuTable { const double* time; const double* rx; const double* ry; const double* rz; int pointer_cur; };

__device__ __forceinline__ RawPoint load_raw(const RawPoint* p, int i) {
    // 24-byte records: three 8-byte loads keep every access naturally aligned
    const uint2* q = reinterpret_cast<const uint2*>(p + i);
    uint2 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
    RawPoint r;
    r.x = __uint_as_float(a.x); r.y = __uint_as_float(a.y); r.z = __uint_as_float(b.x); r.intensity = __uint_as_float(b.y);
    r.ring = (unsigned short)(c.x & 0xffffu); r.pad = 0; r.time = __uint_as_float(c.y);
    return r;
}

__device__ __forceinline__ bool keep_point(const RawPoint& r, int i, const DeskewParams& P) {
    float range = sqrtf(r.x * r.x + r.y * r.y + r.z * r.z);                 // lib/common_lib.cpp:27-31
    if (range < P.lidarMinRange || range > P.lidarMaxRange) return false;   // :581
    int rowIdn = r.ring;
    if (rowIdn < 0 || rowIdn >= P.N_SCAN) return false;                     // :585
    if (rowIdn % P.downsampleRate != 0) return false;                       // :588
    if (i % P.point_filter_num != 0) return false;                          // :591
    return true;
}

__device__ __forceinline__ void find_rotation_dev(double pointTime, const ImuTable& T, float& ox, float& oy, float& oz) {
    int f = 0;
    while (f < T.pointer_cur) { if (pointTime < __ldg(T.time + f)) break; ++f; }           // :497-503 (linear, as the reference)
    const double tf_ = __ldg(T.time + f);
    if (pointTime > tf_ || f == 0) { ox = (float)__ldg(T.rx + f); oy = (float)__ldg(T.ry + f); oz = (float)__ldg(T.rz + f); }   // :505-509
    else {
        const int bk = f - 1; const double tb = __ldg(T.time + bk);
        double ratioFront = (pointTime - tb) / (tf_ - tb);
        double ratioBack = (tf_ - pointTime) / (tf_ - tb);
        ox = (float)(__ldg(T.rx + f) * ratioFront + __ldg(T.rx + bk) * ratioBack);
        oy = (float)(__ldg(T.ry + f) * ratioFront + __ldg(T.ry + bk) * ratioBack);
        oz = (float)(__ldg(T.rz + f) * ratioFront + __ldg(T.rz + bk) * ratioBack);
    }
}

// Eigen::Affine3f::inverse() (3x3 cofactor inverse, translation = -(inv * t))
__device__ __forceinline__ void affine_inverse_dev(const float* t, float* o) {
#define M_(r, c) t[(r) * 4 + (c)]
#define COF_(i, j) (M_(((i) + 1) % 3, ((j) + 1) % 3) * M_(((i) + 2) % 3, ((j) + 2) % 3) - M_(((i) + 1) % 3, ((j) + 2) % 3) * M_(((i) + 2) % 3, ((j) + 1) % 3))
    float c00 = COF_(0, 0), c10 = COF_(1, 0), c20 = COF_(2, 0);
    float det = (c00 * M_(0, 0) + c10 * M_(1, 0)) + c20 * M_(2, 0);
    float invdet = 1.f / det;
    float L[3][3];
    L[0][0] = c00 * invdet; L[0][1] = c10 * invdet; L[0][2] = c20 * invdet;
    L[1][0] = COF_(0, 1) * invdet; L[1][1] = COF_(1, 1) * invdet; L[1][2] = COF_(2, 1) * invdet;
    L[2][0] = COF_(0, 2) * invdet; L[2][1] = COF_(1, 2) * invdet; L[2][2] = COF_(2, 2) * invdet;
#undef COF_
#undef M_
    for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) o[r * 4 + c] = L[r][c];
        o[r * 4 + 3] = -((L[r][0] * t[3] + L[r][1] * t[7]) + L[r][2] * t[11]);
    }
}
__device__ __forceinline__ void affine_mul_dev(const float* a, const float* b, float* o) {
#pragma unroll
    for (int r = 0; r < 3; ++r) {
#pragma unroll
        for (int c = 0; c < 3; ++c) o[r * 4 + c] = (a[r * 4] * b[c] + a[r * 4 + 1] * b[4 + c]) + a[r * 4 + 2] * b[8 + c];
        o[r * 4 + 3] = ((a[r * 4] * b[3] + a[r * 4 + 1] * b[7]) + a[r * 4 + 2] * b[11]) + a[r * 4 + 3];
    }
}

// one block; chunks of blockDim points from the front until a kept point shows up.  Writes transStartInverse (12 floats)
// and first_kept (index or -1).
__global__ void __launch_bounds__(1024) k_first_kept(const RawPoint* __restrict__ raw, int n, DeskewParams P, double timeScanCur, ImuTable T,
                                                    int deskew_enabled, float* __restrict__ start_inv, int* __restrict__ first_kept) {
    __shared__ int s_first;
    if (threadIdx.x == 0) s_first = 0x7fffffff;
    __syncthreads();
    for (int base = 0; base < n; base += blockDim.x) {
        int i = base + threadIdx.x;
        if (i < n) { RawPoint r = load_raw(raw, i); if (keep_point(r, i, P)) atomicMin(&s_first, i); }
        __syncthreads();
        if (s_first != 0x7fffffff) break;
    }
    if (threadIdx.x == 0) {
        int f = s_first == 0x7fffffff ? -1 : s_first;
        *first_kept = f;
        float tf[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};
        if (f >= 0 && deskew_enabled) {
            RawPoint r = load_raw(raw, f);
            float rx, ry, rz; find_rotation_dev(timeScanCur + (double)r.time, T, rx, ry, rz);
            float t0[12]; get_transformation_dev(0.f, 0.f, 0.f, rx, ry, rz, t0);
            affine_inverse_dev(t0, tf);
        }
        for (int k = 0; k < 12; ++k) start_inv[k] = tf[k];
    }
}

struct DeskewLoad {
    const RawPoint* raw; DeskewParams P;
    __device__ __forceinline__ unsigned operator()(int i) const { RawPoint r = load_raw(raw, i); return keep_point(r, i, P) ? 1u : 0u; }
};
struct DeskewStore {                          // compaction only: the ordered list of kept raw indices
    int* kept_index;
    __device__ __forceinline__ void operator()(int i, unsigned v, unsigned excl) const { if (v) kept_index[excl] = i; }
};

// one thread per KEPT point: deskewPoint (:536-566) and the ordered store
__global__ void __launch_bounds__(128) k_deskew_points(const RawPoint* __restrict__ raw, const int* __restrict__ kept_index, const int* __restrict__ n_kept,
                                                      double timeScanCur, ImuTable T, int deskew_enabled, const float* __restrict__ start_inv,
                                                      float4* __restrict__ out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= *n_kept) return;
    const int i = kept_index[k];
    RawPoint r = load_raw(raw, i);
    float4 p = make_float4(r.x, r.y, r.z, r.intensity);
    if (deskew_enabled) {
        float rx, ry, rz; find_rotation_dev(timeScanCur + (double)r.time, T, rx, ry, rz);
        float tf[12]; get_transformation_dev(0.f, 0.f, 0.f, rx, ry, rz, tf);
        float si[12];
#pragma unroll
        for (int q = 0; q < 12; ++q) si[q] = __ldg(start_inv + q);
        float bt[12]; affine_mul_dev(si, tf, bt);
        p = apply_affine_dev(bt, p);
    }
    out[k] = p;
}

struct DeskewWork {
    DevBuf<RawPoint> raw;           // staging for host input
    DevBuf<double> imu;             // 4 x rows (time, rx, ry, rz)
    DevBuf<int> kept;               // ordered raw indices of the kept points
    DevMem<float> start_inv;       // 12 floats
    int* first_kept = nullptr;     // view: a word of the front set's counts
    ScanWork scan;
};

}  // namespace liorf
