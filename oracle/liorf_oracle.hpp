// liorf_oracle.hpp — CPU restatement of liorf's scan-to-map hot path.
//
// THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only tests/, __graft_entry__.smoke()
// and bench.py's cpu_baseline / --impl reference legs may build, link or call it.
// The product (liorf_b200/csrc) never includes this file and has no CPU fallback.
//
// Every function cites the reference file:line it follows (paths relative to the
// jimmyshe/liorf tree).  Where the arithmetic lives in an un-vendored third-party
// library (PCL VoxelGrid / KdTreeFLANN, Eigen ColPivHouseholderQR, OpenCV
// solve/eigen/invert, PCL getTransformation) the published algorithm of that library
// is restated and the header of each block says which upstream routine it follows.
//
// PARITY PINNING (see DESIGN.md §5):
//   * everything that is the REFERENCE'S OWN CODE on the path — control flow, indexing, thresholds, float / double mixes, member state that
//     persists across iterations and frames, call order — is pinned to the reference's own sources compiled UNCHANGED into oracle/_ref/
//     (recipes in oracle/Makefile): include/Scancontext.cpp (oracle/shim), src/mapOptmization.cpp and src/imageProjection.cpp (oracle/shim_ros);
//     tests/test_oracle_vs_reference_sc.py, tests/test_oracle_vs_reference_nodes.py compare bit for bit.
//   * ring-key kNN        — pinned against the reference's own vendored nanoflann 1.3.2 (oracle/_ref/libliorf_ref.so).
//   * 6x6 solve/eigen/inv — pinned against OpenCV 4.13 (python cv2) golden vectors in tests/golden/ (script: tests/golden/make_cv2_golden.py).
//   * PARITY UNPINNED: the ARITHMETIC INSIDE the third-party calls — PCL VoxelGrid / KdTreeFLANN (tie order), Eigen ColPivHouseholderQR and
//     Affine3f inverse / product, PCL getTransformation / getTranslationAndEulerAngles, tf quaternions, Eigen's reduction order in the
//     ScanContext means / norms / dots.  The reference has no tests or golden vectors and PCL / Eigen / tf are not in this container; those
//     blocks follow the upstream algorithms as documented, and the header stand-ins the reference sources are compiled against forward to
//     exactly these blocks (so the comparisons above hold GIVEN these kernels).
//
// Plain C++17, no dependencies.  Compiled WITHOUT FMA contraction (-ffp-contract=off)
// and without -march, like the reference build (CMakeLists.txt:7).
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>
#include <numeric>
#include <utility>
#include <vector>
#include <deque>

namespace liorf_oracle {

struct P4 { float x, y, z, i; };                    // pcl::PointXYZI payload (include/utility.h:61)
struct PRaw { float x, y, z, i; uint16_t ring; uint16_t pad; float time; };  // src/imageProjection.cpp:4-15

// ------------------------------------------------------------------------------------------------
// T — pcl::getTransformation(x,y,z,roll,pitch,yaw) (float Scalar); row-major 3x4.
// Used at src/mapOptmization.cpp:317,350 and src/imageProjection.cpp:551,556.
// ------------------------------------------------------------------------------------------------
inline void get_transformation(float x, float y, float z, float roll, float pitch, float yaw, float t[12]) {
    float A = std::cos(yaw), B = std::sin(yaw), C = std::cos(pitch), D = std::sin(pitch);
    float E = std::cos(roll), F = std::sin(roll), DE = D * E, DF = D * F;
    t[0] = A * C;  t[1] = A * DF - B * E;  t[2]  = B * F + A * DE;  t[3]  = x;
    t[4] = B * C;  t[5] = A * E + B * DF;  t[6]  = B * DE - A * F;  t[7]  = y;
    t[8] = -D;     t[9] = C * F;           t[10] = C * E;           t[11] = z;
}
// trans2Affine3f (src/mapOptmization.cpp:348-351): transformIn = (roll,pitch,yaw,x,y,z)
inline void trans2affine(const float tf[6], float t[12]) { get_transformation(tf[3], tf[4], tf[5], tf[0], tf[1], tf[2], t); }

// pointAssociateToMap / transformPointCloud op order (src/mapOptmization.cpp:304-306, 323-325)
inline P4 apply_affine(const float t[12], const P4& p) {
    P4 o;
    o.x = t[0] * p.x + t[1] * p.y + t[2]  * p.z + t[3];
    o.y = t[4] * p.x + t[5] * p.y + t[6]  * p.z + t[7];
    o.z = t[8] * p.x + t[9] * p.y + t[10] * p.z + t[11];
    o.i = p.i;
    return o;
}

// ------------------------------------------------------------------------------------------------
// V — pcl::VoxelGrid<PointXYZI>::applyFilter (downsample_all_data_=true, min_points_per_voxel_=0)
// call sites src/mapOptmization.cpp:1037-1038 (local map), 1064-1065 (current scan).
// Returns number of output points, or -1 when PCL's int32 index overflow guard fires (PCL then
// copies the input through unfiltered).  membership[i] = output slot of input point i.
// Voxel order: PCL's, ascending unsigned index (wrapped mod 2^32).  Canonical rule for the unspecified (unstable-sort)
// intra-voxel order: ascending input index.
// ------------------------------------------------------------------------------------------------
struct VoxelMeta { float minp[3], maxp[3]; int min_b[3], div_b[3]; float inv_leaf; };

inline int voxel_grid(const P4* in, int n, float leaf, std::vector<P4>& out, std::vector<int>* membership = nullptr,
                      std::vector<int>* out_keys = nullptr, VoxelMeta* meta = nullptr) {
    out.clear();
    if (membership) membership->assign(n, -1);
    if (out_keys) out_keys->clear();
    if (n == 0) return 0;
    float mn[3] = {in[0].x, in[0].y, in[0].z}, mx[3] = {in[0].x, in[0].y, in[0].z};
    for (int k = 1; k < n; ++k) {               // pcl::getMinMax3D
        mn[0] = std::min(mn[0], in[k].x); mx[0] = std::max(mx[0], in[k].x);
        mn[1] = std::min(mn[1], in[k].y); mx[1] = std::max(mx[1], in[k].y);
        mn[2] = std::min(mn[2], in[k].z); mx[2] = std::max(mx[2], in[k].z);
    }
    const float inv = 1.0f / leaf;              // inverse_leaf_size_ = Ones / leaf_size_
    int64_t dx = (int64_t)((mx[0] - mn[0]) * inv) + 1, dy = (int64_t)((mx[1] - mn[1]) * inv) + 1,
            dz = (int64_t)((mx[2] - mn[2]) * inv) + 1;
    int min_b[3], max_b[3], div_b[3];
    for (int a = 0; a < 3; ++a) {
        min_b[a] = (int)std::floor(mn[a] * inv);
        max_b[a] = (int)std::floor(mx[a] * inv);
        div_b[a] = max_b[a] - min_b[a] + 1;
    }
    if (meta) { for (int a = 0; a < 3; ++a) { meta->minp[a] = mn[a]; meta->maxp[a] = mx[a]; meta->min_b[a] = min_b[a]; meta->div_b[a] = div_b[a]; } meta->inv_leaf = inv; }
    if (dx * dy * dz > (int64_t)std::numeric_limits<int32_t>::max()) return -1;   // "Leaf size is too small"
    // The guard bounds dx·dy·dz, but the index uses div_b, which can be one larger per axis: indices can pass 2^31 and even 2^32.
    // PCL computes the index in int (wrapping) and stores it as unsigned int; cloud_point_index_idx::operator< compares unsigned.
    const int64_t mul1 = div_b[0], mul2 = (int64_t)div_b[0] * div_b[1];
    std::vector<std::pair<uint32_t, int>> iv(n);     // (voxel idx mod 2^32, point index)
    for (int k = 0; k < n; ++k) {
        int i0 = (int)(std::floor(in[k].x * inv) - (float)min_b[0]);
        int i1 = (int)(std::floor(in[k].y * inv) - (float)min_b[1]);
        int i2 = (int)(std::floor(in[k].z * inv) - (float)min_b[2]);
        iv[k] = {(uint32_t)(i0 + i1 * mul1 + i2 * mul2), k};
    }
    std::sort(iv.begin(), iv.end());            // (unsigned idx, point index) lexicographic == stable by idx
    int k = 0;
    while (k < n) {
        int j = k;
        float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f;
        while (j < n && iv[j].first == iv[k].first) {
            const P4& p = in[iv[j].second];
            sx += p.x; sy += p.y; sz += p.z; si += p.i;
            if (membership) (*membership)[iv[j].second] = (int)out.size();
            ++j;
        }
        float cnt = (float)(j - k);
        out.push_back(P4{sx / cnt, sy / cnt, sz / cnt, si / cnt});
        if (out_keys) out_keys->push_back((int)iv[k].first);     // the int32 bit pattern of the unsigned index
        k = j;
    }
    return (int)out.size();
}

// ------------------------------------------------------------------------------------------------
// N — exact 5-NN, FLANN L2_Simple distance in fp32: d = dx*dx; d += dy*dy; d += dz*dz.
// call site src/mapOptmization.cpp:1087.  Canonical tie-break (distance, index).  Brute force.
// ------------------------------------------------------------------------------------------------
inline float l2_simple3(const P4& a, const P4& b) {
    float dx = a.x - b.x, dy = a.y - b.y, dz = a.z - b.z;
    float d = dx * dx; d += dy * dy; d += dz * dz;
    return d;
}
inline void knn5_brute(const P4* map, int m, const P4& q, int idx[5], float d2[5]) {
    for (int j = 0; j < 5; ++j) { idx[j] = -1; d2[j] = std::numeric_limits<float>::infinity(); }
    for (int k = 0; k < m; ++k) {
        float d = l2_simple3(q, map[k]);
        if (d > d2[4] || (d == d2[4] && idx[4] >= 0)) continue;  // ascending k ⇒ ties keep the lower index
        int j = 4;
        while (j > 0 && (d2[j - 1] > d)) { d2[j] = d2[j - 1]; idx[j] = idx[j - 1]; --j; }
        d2[j] = d; idx[j] = k;
    }
}

// ------------------------------------------------------------------------------------------------
// Q — Eigen::ColPivHouseholderQR<Matrix<float,5,3>>::solve (Eigen 3.3 computeInPlace / _solve_impl,
// LAPACK-style column-norm downdating), call site src/mapOptmization.cpp:1104.
// A is 5x3 row-major, b is 5x1; x = argmin ||A x - b||.  Sequential fp32 reductions.
// ------------------------------------------------------------------------------------------------
inline void colpiv_qr_solve_5x3(const float Ain[15], const float bin[5], float x[3]) {
    const int R = 5, C = 3;
    float qr[5][3];
    for (int r = 0; r < R; ++r) for (int c = 0; c < C; ++c) qr[r][c] = Ain[r * 3 + c];
    float hcoef[3], normsUpd[3], normsDir[3];
    int perm[3] = {0, 1, 2}, transp[3];
    for (int c = 0; c < C; ++c) {
        float s = 0.f; for (int r = 0; r < R; ++r) s += qr[r][c] * qr[r][c];
        normsDir[c] = normsUpd[c] = std::sqrt(s);
    }
    const float eps = std::numeric_limits<float>::epsilon();
    float maxn = std::max(normsUpd[0], std::max(normsUpd[1], normsUpd[2]));
    float th = maxn * eps / (float)R; const float threshold_helper = th * th;
    const float norm_downdate_threshold = std::sqrt(eps);
    int nonzero_pivots = C;
    for (int k = 0; k < C; ++k) {
        int big = k; float bign = normsUpd[k];
        for (int c = k + 1; c < C; ++c) if (normsUpd[c] > bign) { bign = normsUpd[c]; big = c; }
        float big_sq = bign * bign;
        if (nonzero_pivots == C && big_sq < threshold_helper * (float)(R - k)) nonzero_pivots = k;
        transp[k] = big;
        if (k != big) {
            for (int r = 0; r < R; ++r) std::swap(qr[r][k], qr[r][big]);
            std::swap(normsUpd[k], normsUpd[big]); std::swap(normsDir[k], normsDir[big]);
        }
        // makeHouseholderInPlace on qr.col(k).tail(R-k)
        float tailSq = 0.f; for (int r = k + 1; r < R; ++r) tailSq += qr[r][k] * qr[r][k];
        float c0 = qr[k][k], beta, tau;
        if (tailSq <= std::numeric_limits<float>::min()) {
            tau = 0.f; beta = c0; for (int r = k + 1; r < R; ++r) qr[r][k] = 0.f;
        } else {
            beta = std::sqrt(c0 * c0 + tailSq);
            if (c0 >= 0.f) beta = -beta;
            float den = c0 - beta;
            for (int r = k + 1; r < R; ++r) qr[r][k] = qr[r][k] / den;
            tau = (beta - c0) / beta;
        }
        hcoef[k] = tau; qr[k][k] = beta;
        // applyHouseholderOnTheLeft to bottomRightCorner(R-k, C-k-1)
        if (tau != 0.f) {
            for (int c = k + 1; c < C; ++c) {
                float tmp = 0.f; for (int r = k + 1; r < R; ++r) tmp += qr[r][k] * qr[r][c];
                tmp += qr[k][c];
                qr[k][c] -= tau * tmp;
                for (int r = k + 1; r < R; ++r) qr[r][c] -= (tau * qr[r][k]) * tmp;
            }
        }
        for (int c = k + 1; c < C; ++c) {
            if (normsUpd[c] != 0.f) {
                float temp = std::fabs(qr[k][c]) / normsUpd[c];
                temp = (1.f + temp) * (1.f - temp);
                temp = temp < 0.f ? 0.f : temp;
                float ratio = normsUpd[c] / normsDir[c];
                float temp2 = temp * (ratio * ratio);
                if (temp2 <= norm_downdate_threshold) {
                    float s = 0.f; for (int r = k + 1; r < R; ++r) s += qr[r][c] * qr[r][c];
                    normsDir[c] = std::sqrt(s); normsUpd[c] = normsDir[c];
                } else normsUpd[c] *= std::sqrt(temp);
            }
        }
    }
    for (int k = 0; k < C; ++k) std::swap(perm[k], perm[transp[k]]);   // PermutationMatrix from transpositions
    // Eigen builds the permutation as P = T0*T1*...; applyTranspositionOnTheRight(k, transp[k]) for k ascending
    // which swaps indices[k] and indices[transp[k]] — as done above.
    float c[5]; for (int r = 0; r < R; ++r) c[r] = bin[r];
    for (int k = 0; k < nonzero_pivots; ++k) {      // c = H_k ... H_0 b  (householderQ().adjoint())
        float tau = hcoef[k];
        if (tau == 0.f) continue;
        float tmp = 0.f; for (int r = k + 1; r < R; ++r) tmp += qr[r][k] * c[r];
        tmp += c[k];
        c[k] -= tau * tmp;
        for (int r = k + 1; r < R; ++r) c[r] -= (tau * qr[r][k]) * tmp;
    }
    x[0] = x[1] = x[2] = 0.f;
    if (nonzero_pivots == 0) return;
    for (int i = nonzero_pivots - 1; i >= 0; --i) {   // upper-triangular back substitution
        float s = c[i];
        for (int j = i + 1; j < nonzero_pivots; ++j) s -= qr[i][j] * c[j];
        c[i] = s / qr[i][i];
    }
    for (int i = 0; i < nonzero_pivots; ++i) x[perm[i]] = c[i];
}

// ------------------------------------------------------------------------------------------------
// a7 — surfOptimization body for one point (src/mapOptmization.cpp:1079-1142), given the
// neighbour set.  Returns flag (laserCloudOriSurfFlag[i]).
// ------------------------------------------------------------------------------------------------
inline bool surf_point(const P4& pointOri, const P4& pointSel, const P4* map, const int idx[5], const float d2[5],
                       P4& coeff, float plane[4] = nullptr) {
    coeff = P4{0, 0, 0, 0};
    if (idx[4] < 0 || !(d2[4] < 1.0)) return false;                  // :1097
    float A[15], b[5], x[3];
    for (int j = 0; j < 5; ++j) { A[j * 3] = map[idx[j]].x; A[j * 3 + 1] = map[idx[j]].y; A[j * 3 + 2] = map[idx[j]].z; b[j] = -1.f; }
    colpiv_qr_solve_5x3(A, b, x);                                      // :1104
    float pa = x[0], pb = x[1], pc = x[2], pd = 1.f;
    float ps = std::sqrt(pa * pa + pb * pb + pc * pc);                 // :1111
    pa /= ps; pb /= ps; pc /= ps; pd /= ps;
    if (plane) { plane[0] = pa; plane[1] = pb; plane[2] = pc; plane[3] = pd; }
    for (int j = 0; j < 5; ++j) {                                      // :1115-1122
        const P4& m = map[idx[j]];
        if (std::fabs(pa * m.x + pb * m.y + pc * m.z + pd) > 0.2) return false;
    }
    float pd2 = pa * pointSel.x + pb * pointSel.y + pc * pointSel.z + pd;   // :1125
    // :1127-1128 — double expression (0.9 is a double literal), float sqrt(sqrt(.)) of a float sum
    float s = (float)(1 - 0.9 * std::fabs(pd2) /
                      std::sqrt(std::sqrt(pointOri.x * pointOri.x + pointOri.y * pointOri.y + pointOri.z * pointOri.z)));
    coeff.x = s * pa; coeff.y = s * pb; coeff.z = s * pc; coeff.i = s * pd2;   // :1130-1133
    return s > 0.1;                                                    // :1135
}

// ------------------------------------------------------------------------------------------------
// OpenCV core restatements used by LMOptimization (src/mapOptmization.cpp:1237-1271), float.
//   qr_solve  = cv::solve(..., DECOMP_QR)  → hal::QR32f / QRImpl (modules/core/src/lapack.cpp)
//   jacobi    = cv::eigen                  → JacobiImpl_<float>, eigenvalues descending, rows of V
//   lu_invert = cv::Mat::inv() DECOMP_LU   → hal::LU32f / LUImpl on [A | I]
//   gemm6     = cv::gemm small-matrix path: double accumulator, rounded to float
// ------------------------------------------------------------------------------------------------
inline bool cv_qr_solve6(const float Ain[36], const float bin[6], float x[6]) {
    const int m = 6, n = 6;
    float A[36], b[6], vl[6], hF[6];
    std::memcpy(A, Ain, sizeof(A)); std::memcpy(b, bin, sizeof(b));
    for (int l = 0; l < n; ++l) {
        int vlSize = m - l; float vlNorm = 0.f;
        for (int i = 0; i < vlSize; ++i) { vl[i] = A[(l + i) * 6 + l]; vlNorm += vl[i] * vl[i]; }
        float tmpV = vl[0];
        vl[0] = vl[0] + (vl[0] < 0.f ? -1.f : 1.f) * std::sqrt(vlNorm);
        vlNorm = std::sqrt(vlNorm + vl[0] * vl[0] - tmpV * tmpV);
        for (int i = 0; i < vlSize; ++i) vl[i] /= vlNorm;
        for (int j = l; j < n; ++j) {
            float v_lA = 0.f;
            for (int i = l; i < m; ++i) v_lA += vl[i - l] * A[i * 6 + j];
            for (int i = l; i < m; ++i) A[i * 6 + j] -= 2 * vl[i - l] * v_lA;
        }
        hF[l] = vl[0] * vl[0];
        for (int i = 1; i < vlSize; ++i) A[(l + i) * 6 + l] = vl[i] / vl[0];
    }
    for (int l = 0; l < n; ++l) {
        vl[0] = 1.f;
        for (int j = 1; j < m - l; ++j) vl[j] = A[(j + l) * 6 + l];
        float v_lB = 0.f;
        for (int i = l; i < m; ++i) v_lB += vl[i - l] * b[i];
        for (int i = l; i < m; ++i) b[i] -= 2 * vl[i - l] * v_lB * hF[l];
    }
    const float eps = std::numeric_limits<float>::epsilon() * 10;   // hal::QR32f passes FLT_EPSILON*10
    for (int i = n - 1; i >= 0; --i) {
        for (int j = n - 1; j > i; --j) b[i] -= b[j] * A[i * 6 + j];
        if (std::fabs(A[i * 6 + i]) < eps) { for (int k = 0; k < 6; ++k) x[k] = 0.f; return false; }
        b[i] /= A[i * 6 + i];
    }
    std::memcpy(x, b, sizeof(b));
    return true;
}

inline float cv_hypot(float a, float b) {
    a = std::fabs(a); b = std::fabs(b);
    if (a > b) { b /= a; return a * std::sqrt(1 + b * b); }
    if (b > 0) { a /= b; return b * std::sqrt(1 + a * a); }
    return 0.f;
}

// W[6] eigenvalues descending, V 6x6 row-major with eigenvectors in ROWS.
inline void cv_jacobi6(const float Ain[36], float W[6], float V[36]) {
    const int n = 6; const float eps = std::numeric_limits<float>::epsilon();
    float A[36]; std::memcpy(A, Ain, sizeof(A));
    int indR[6], indC[6]; int i, j, k, m; float mv;
    for (i = 0; i < n; ++i) { for (j = 0; j < n; ++j) V[i * 6 + j] = 0.f; V[i * 6 + i] = 1.f; }
    for (k = 0; k < n; ++k) {
        W[k] = A[7 * k];
        if (k < n - 1) {
            for (m = k + 1, mv = std::fabs(A[6 * k + m]), i = k + 2; i < n; ++i) { float val = std::fabs(A[6 * k + i]); if (mv < val) mv = val, m = i; }
            indR[k] = m;
        }
        if (k > 0) {
            for (m = 0, mv = std::fabs(A[k]), i = 1; i < k; ++i) { float val = std::fabs(A[6 * i + k]); if (mv < val) mv = val, m = i; }
            indC[k] = m;
        }
    }
    const int maxIters = n * n * 30;
    for (int iters = 0; iters < maxIters; ++iters) {
        for (k = 0, mv = std::fabs(A[indR[0]]), i = 1; i < n - 1; ++i) { float val = std::fabs(A[6 * i + indR[i]]); if (mv < val) mv = val, k = i; }
        int l = indR[k];
        for (i = 1; i < n; ++i) { float val = std::fabs(A[6 * indC[i] + i]); if (mv < val) mv = val, k = indC[i], l = i; }
        float p = A[6 * k + l];
        if (std::fabs(p) <= eps) break;
        float y = (float)((W[l] - W[k]) * 0.5);
        float t = std::fabs(y) + cv_hypot(p, y);
        float s = cv_hypot(p, t);
        float c = t / s;
        s = p / s; t = (p / t) * p;
        if (y < 0) s = -s, t = -t;
        A[6 * k + l] = 0;
        W[k] -= t; W[l] += t;
        float a0, b0;
#define LIORF_ROT(v0, v1) a0 = v0, b0 = v1, v0 = a0 * c - b0 * s, v1 = a0 * s + b0 * c
        for (i = 0; i < k; ++i) LIORF_ROT(A[6 * i + k], A[6 * i + l]);
        for (i = k + 1; i < l; ++i) LIORF_ROT(A[6 * k + i], A[6 * i + l]);
        for (i = l + 1; i < n; ++i) LIORF_ROT(A[6 * k + i], A[6 * l + i]);
        for (i = 0; i < n; ++i) LIORF_ROT(V[6 * k + i], V[6 * l + i]);
#undef LIORF_ROT
        for (j = 0; j < 2; ++j) {
            int idx = j == 0 ? k : l;
            if (idx < n - 1) {
                for (m = idx + 1, mv = std::fabs(A[6 * idx + m]), i = idx + 2; i < n; ++i) { float val = std::fabs(A[6 * idx + i]); if (mv < val) mv = val, m = i; }
                indR[idx] = m;
            }
            if (idx > 0) {
                for (m = 0, mv = std::fabs(A[idx]), i = 1; i < idx; ++i) { float val = std::fabs(A[6 * i + idx]); if (mv < val) mv = val, m = i; }
                indC[idx] = m;
            }
        }
    }
    for (k = 0; k < n - 1; ++k) {
        m = k;
        for (i = k + 1; i < n; ++i) if (W[m] < W[i]) m = i;
        if (k != m) { std::swap(W[m], W[k]); for (i = 0; i < n; ++i) std::swap(V[6 * m + i], V[6 * k + i]); }
    }
}

inline bool cv_lu_invert6(const float Ain[36], float inv[36]) {
    const int m = 6; float A[36]; std::memcpy(A, Ain, sizeof(A));
    for (int i = 0; i < 36; ++i) inv[i] = 0.f;
    for (int i = 0; i < 6; ++i) inv[i * 6 + i] = 1.f;
    const float eps = std::numeric_limits<float>::epsilon() * 10;
    for (int i = 0; i < m; ++i) {
        int k = i;
        for (int j = i + 1; j < m; ++j) if (std::fabs(A[j * 6 + i]) > std::fabs(A[k * 6 + i])) k = j;
        if (std::fabs(A[k * 6 + i]) < eps) { for (int q = 0; q < 36; ++q) inv[q] = 0.f; return false; }
        if (k != i) {
            for (int j = i; j < m; ++j) std::swap(A[i * 6 + j], A[k * 6 + j]);
            for (int j = 0; j < m; ++j) std::swap(inv[i * 6 + j], inv[k * 6 + j]);
        }
        float d = -1 / A[i * 6 + i];
        for (int j = i + 1; j < m; ++j) {
            float alpha = A[j * 6 + i] * d;
            for (int q = i + 1; q < m; ++q) A[j * 6 + q] += alpha * A[i * 6 + q];
            for (int q = 0; q < m; ++q) inv[j * 6 + q] += alpha * inv[i * 6 + q];
        }
    }
    for (int i = m - 1; i >= 0; --i)
        for (int j = 0; j < m; ++j) {
            float s = inv[i * 6 + j];
            for (int k = i + 1; k < m; ++k) s -= A[i * 6 + k] * inv[k * 6 + j];
            inv[i * 6 + j] = s / A[i * 6 + i];
        }
    return true;
}

inline void cv_gemm6(const float A[36], const float B[36], float Cc[36]) {     // double accumulator
    for (int i = 0; i < 6; ++i) for (int j = 0; j < 6; ++j) {
        double s = 0; for (int k = 0; k < 6; ++k) s += (double)A[i * 6 + k] * (double)B[k * 6 + j];
        Cc[i * 6 + j] = (float)s;
    }
}
inline void cv_gemv6(const float A[36], const float x[6], float y[6]) {
    for (int i = 0; i < 6; ++i) { double s = 0; for (int k = 0; k < 6; ++k) s += (double)A[i * 6 + k] * (double)x[k]; y[i] = (float)s; }
}

// ------------------------------------------------------------------------------------------------
// a9 — LMOptimization (src/mapOptmization.cpp:1158-1293).  State that persists across iterations and
// frames (isDegenerate, matP: members at :139-140) lives in LMState.
// ------------------------------------------------------------------------------------------------
struct LMState { bool isDegenerate = false; float matP[36] = {0}; };

inline void lm_row(const float tf[6], const P4& p, const P4& c, float row[6], float& b) {
    float srx = std::sin(tf[2]), crx = std::cos(tf[2]);          // :1170-1175 (yaw, pitch, roll)
    float sry = std::sin(tf[1]), cry = std::cos(tf[1]);
    float srz = std::sin(tf[0]), crz = std::cos(tf[0]);
    float arx = (-srx * cry * p.x - (srx * sry * srz + crx * crz) * p.y + (crx * srz - srx * sry * crz) * p.z) * c.x
              + (crx * cry * p.x - (srx * crz - crx * sry * srz) * p.y + (crx * sry * crz + srx * srz) * p.z) * c.y;
    float ary = (-crx * sry * p.x + crx * cry * srz * p.y + crx * cry * crz * p.z) * c.x
              + (-srx * sry * p.x + srx * sry * srz * p.y + srx * cry * crz * p.z) * c.y
              + (-cry * p.x - sry * srz * p.y - sry * crz * p.z) * c.z;
    float arz = ((crx * sry * crz + srx * srz) * p.y + (srx * crz - crx * sry * srz) * p.z) * c.x
              + ((-crx * srz + srx * sry * crz) * p.y + (-srx * sry * srz - crx * crz) * p.z) * c.y
              + (cry * crz * p.y - cry * srz * p.z) * c.z;
    row[0] = arz; row[1] = ary; row[2] = arx; row[3] = c.x; row[4] = c.y; row[5] = c.z;   // :1228-1233
    b = -c.i;                                                                          // :1234
}

struct LMTrace { float AtA[36]; float AtB[6]; float X[6]; int nsel; int converged; int degenerate; int solved; };

// returns true when converged (:1289-1291).  tf is transformTobeMapped (roll,pitch,yaw,x,y,z).
inline bool lm_optimization(int iterCount, const P4* ori, const P4* coeff, int nsel, float tf[6], LMState& st, LMTrace* tr = nullptr) {
    if (tr) { std::memset(tr, 0, sizeof(*tr)); tr->nsel = nsel; tr->degenerate = st.isDegenerate; }
    if (nsel < 50) return false;                                               // :1178
    double acc[6][6] = {{0}}, accb[6] = {0};
    for (int i = 0; i < nsel; ++i) {                                           // matAt*matA, matAt*matB (:1237-1239)
        float r[6], b; lm_row(tf, ori[i], coeff[i], r, b);
        for (int a = 0; a < 6; ++a) { for (int c = 0; c < 6; ++c) acc[a][c] += (double)r[a] * (double)r[c]; accb[a] += (double)r[a] * (double)b; }
    }
    float AtA[36], AtB[6], X[6];
    for (int a = 0; a < 6; ++a) { for (int c = 0; c < 6; ++c) AtA[a * 6 + c] = (float)acc[a][c]; AtB[a] = (float)accb[a]; }
    bool solved = cv_qr_solve6(AtA, AtB, X);                                   // :1240
    if (iterCount == 0) {                                                      // :1242-1264
        float E[6], V[36], V2[36];
        cv_jacobi6(AtA, E, V);
        std::memcpy(V2, V, sizeof(V));
        st.isDegenerate = false;
        for (int i = 5; i >= 0; --i) {
            if (E[i] < 100.f) { for (int j = 0; j < 6; ++j) V2[i * 6 + j] = 0.f; st.isDegenerate = true; }
            else break;
        }
        float Vinv[36]; cv_lu_invert6(V, Vinv);
        cv_gemm6(Vinv, V2, st.matP);
    }
    if (st.isDegenerate) { float X2[6]; std::memcpy(X2, X, sizeof(X)); cv_gemv6(st.matP, X2, X); }   // :1266-1271
    for (int a = 0; a < 6; ++a) tf[a] += X[a];                                 // :1273-1278
    const float r2d = 57.29578f;                                                // pcl::rad2deg(float) = alpha * 57.29578f
    // pow(float,int) promotes to double (C++11); the sum and sqrt are double, the result is stored to float (:1280-1287)
    float deltaR = (float)std::sqrt(std::pow((double)(X[0] * r2d), 2) + std::pow((double)(X[1] * r2d), 2) + std::pow((double)(X[2] * r2d), 2));
    float deltaT = (float)std::sqrt(std::pow((double)(X[3] * 100), 2) + std::pow((double)(X[4] * 100), 2) + std::pow((double)(X[5] * 100), 2));
    bool conv = deltaR < 0.05 && deltaT < 0.05;                                // :1289
    if (tr) { std::memcpy(tr->AtA, AtA, sizeof(AtA)); std::memcpy(tr->AtB, AtB, sizeof(AtB)); std::memcpy(tr->X, X, sizeof(X));
              tr->converged = conv; tr->degenerate = st.isDegenerate; tr->solved = solved; }
    return conv;
}

// ------------------------------------------------------------------------------------------------
// a1/a2 — projectPointCloud + deskewPoint + findRotation (src/imageProjection.cpp:493-598)
// ------------------------------------------------------------------------------------------------
struct DeskewParams { float lidarMinRange, lidarMaxRange; int N_SCAN, downsampleRate, point_filter_num; };

// imuDeskewInfo (src/imageProjection.cpp:350-409) restated over a std::deque like the reference's imuQueue (pop_front and all).
// sample = {stamp, wx, wy, wz}; returns imuAvailable, fills the tables (sized queueLength = 2000, :62) and imuPointerCur.
struct ImuSample { double stamp, wx, wy, wz; };
inline bool imu_deskew_info(std::deque<ImuSample>& imuQueue, double timeScanCur, double timeScanEnd, std::vector<double>& imuTime,
                            std::vector<double>& imuRotX, std::vector<double>& imuRotY, std::vector<double>& imuRotZ, int& imuPointerCur) {
    bool imuAvailable = false;
    while (!imuQueue.empty()) {                                           // :354-360
        if (imuQueue.front().stamp < timeScanCur - 0.01) imuQueue.pop_front();
        else break;
    }
    if (imuQueue.empty()) return imuAvailable;                            // :362-363
    imuPointerCur = 0;                                                    // :365
    for (int i = 0; i < (int)imuQueue.size(); ++i) {                      // :367
        const ImuSample thisImuMsg = imuQueue[i];
        const double currentImuTime = thisImuMsg.stamp;
        if (currentImuTime > timeScanEnd + 0.01) break;                   // :378-379
        if (imuPointerCur == 0) {                                         // :381-388
            imuRotX[0] = 0; imuRotY[0] = 0; imuRotZ[0] = 0; imuTime[0] = currentImuTime;
            ++imuPointerCur;
            continue;
        }
        const double timeDiff = currentImuTime - imuTime[imuPointerCur - 1];                        // :395
        imuRotX[imuPointerCur] = imuRotX[imuPointerCur - 1] + thisImuMsg.wx * timeDiff;            // :396-398
        imuRotY[imuPointerCur] = imuRotY[imuPointerCur - 1] + thisImuMsg.wy * timeDiff;
        imuRotZ[imuPointerCur] = imuRotZ[imuPointerCur - 1] + thisImuMsg.wz * timeDiff;
        imuTime[imuPointerCur] = currentImuTime;
        ++imuPointerCur;
    }
    --imuPointerCur;                                                      // :403
    if (imuPointerCur <= 0) return imuAvailable;                          // :405-406
    imuAvailable = true;
    return imuAvailable;
}

inline void find_rotation(double pointTime, const double* imuTime, const double* rx, const double* ry, const double* rz,
                          int imuPointerCur, float* ox, float* oy, float* oz) {
    *ox = 0; *oy = 0; *oz = 0;
    int f = 0;
    while (f < imuPointerCur) { if (pointTime < imuTime[f]) break; ++f; }          // :497-503
    if (pointTime > imuTime[f] || f == 0) { *ox = (float)rx[f]; *oy = (float)ry[f]; *oz = (float)rz[f]; }  // :505-509
    else {
        int bk = f - 1;
        double ratioFront = (pointTime - imuTime[bk]) / (imuTime[f] - imuTime[bk]);
        double ratioBack = (imuTime[f] - pointTime) / (imuTime[f] - imuTime[bk]);
        *ox = (float)(rx[f] * ratioFront + rx[bk] * ratioBack);
        *oy = (float)(ry[f] * ratioFront + ry[bk] * ratioBack);
        *oz = (float)(rz[f] * ratioFront + rz[bk] * ratioBack);
    }
}

// Eigen::Affine3f::inverse() (Affine mode): linear part by the 3x3 cofactor formula
// (Eigen/src/LU/InverseImpl.h compute_inverse_size3_helper), translation = -(inv * t).
inline void affine_inverse(const float t[12], float o[12]) {
    auto M = [&](int r, int c) { return t[r * 4 + c]; };
    auto cof = [&](int i, int j) {
        int i1 = (i + 1) % 3, i2 = (i + 2) % 3, j1 = (j + 1) % 3, j2 = (j + 2) % 3;
        return M(i1, j1) * M(i2, j2) - M(i1, j2) * M(i2, j1);
    };
    float c00 = cof(0, 0), c10 = cof(1, 0), c20 = cof(2, 0);
    float det = (c00 * M(0, 0) + c10 * M(1, 0)) + c20 * M(2, 0);
    float invdet = 1.f / det;
    float L[3][3];
    L[0][0] = c00 * invdet; L[0][1] = c10 * invdet; L[0][2] = c20 * invdet;
    L[1][0] = cof(0, 1) * invdet; L[1][1] = cof(1, 1) * invdet; L[1][2] = cof(2, 1) * invdet;
    L[2][0] = cof(0, 2) * invdet; L[2][1] = cof(1, 2) * invdet; L[2][2] = cof(2, 2) * invdet;
    for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) o[r * 4 + c] = L[r][c];
        o[r * 4 + 3] = -((L[r][0] * t[3] + L[r][1] * t[7]) + L[r][2] * t[11]);
    }
}
// Affine3f * Affine3f: linear = La*Lb, translation = La*tb + ta (coefficient-wise, k ascending)
inline void affine_mul(const float a[12], const float b[12], float o[12]) {
    for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) o[r * 4 + c] = (a[r * 4] * b[c] + a[r * 4 + 1] * b[4 + c]) + a[r * 4 + 2] * b[8 + c];
        o[r * 4 + 3] = ((a[r * 4] * b[3] + a[r * 4 + 1] * b[7]) + a[r * 4 + 2] * b[11]) + a[r * 4 + 3];
    }
}


// ---------------------------------------------------------------------------------------------------------------------
// updateInitialGuess (src/mapOptmization.cpp:899-958) and transformUpdate (:1323-1353), scalar host code in the reference.
// Restated as one object holding what the reference keeps in members / function-local statics.  tf::Quaternion and
// tf::Matrix3x3 (ROS tf, tfScalar = double; not in this container → parity unpinned) are restated from their published
// formulas: setRPY, angleShortestPath, slerp, Matrix3x3::setRotation + getEulerYPR.
// ---------------------------------------------------------------------------------------------------------------------
struct GuessCloudInfo { int imuAvailable, odomAvailable; float imuRollInit, imuPitchInit, imuYawInit, gx, gy, gz, groll, gpitch, gyaw; };
struct MapOptScalarState {
    float transformTobeMapped[6] = {0, 0, 0, 0, 0, 0};
    float lastImuTransformation[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};
    float lastImuPreTransformation[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};
    int lastImuPreTransAvailable = 0;

    void euler_of(const float t[12]) {                                          // pcl::getTranslationAndEulerAngles into transformTobeMapped
        transformTobeMapped[3] = t[3]; transformTobeMapped[4] = t[7]; transformTobeMapped[5] = t[11];
        transformTobeMapped[0] = std::atan2(t[9], t[10]); transformTobeMapped[1] = std::asin(-t[8]); transformTobeMapped[2] = std::atan2(t[4], t[0]);
    }
    void advance_by(const float last[12], const float now[12]) {                 // transTobe * (last^-1 * now)
        float li[12], inc[12], tobe[12], fin[12];
        affine_inverse(last, li); affine_mul(li, now, inc);
        trans2affine(transformTobeMapped, tobe); affine_mul(tobe, inc, fin);
        euler_of(fin);
    }
    void updateInitialGuess(bool cloudKeyPoses3D_empty, const GuessCloudInfo& ci, bool useImuHeadingInitialization, int imuType) {
        float imuNow[12]; get_transformation(0, 0, 0, ci.imuRollInit, ci.imuPitchInit, ci.imuYawInit, imuNow);
        if (cloudKeyPoses3D_empty) {                                             // :906-917
            transformTobeMapped[0] = ci.imuRollInit; transformTobeMapped[1] = ci.imuPitchInit;
            transformTobeMapped[2] = useImuHeadingInitialization ? ci.imuYawInit : 0.f;
            std::memcpy(lastImuTransformation, imuNow, sizeof(imuNow));
            return;
        }
        if (ci.odomAvailable) {                                                  // :922
            float transBack[12]; get_transformation(ci.gx, ci.gy, ci.gz, ci.groll, ci.gpitch, ci.gyaw, transBack);
            const bool first = !lastImuPreTransAvailable;
            if (!first) advance_by(lastImuPreTransformation, transBack);         // :932-936
            std::memcpy(lastImuPreTransformation, transBack, sizeof(transBack)); lastImuPreTransAvailable = 1;
            if (!first) { std::memcpy(lastImuTransformation, imuNow, sizeof(imuNow)); return; }   // :940-941
        }
        if (ci.imuAvailable && imuType) {                                        // :946-957
            advance_by(lastImuTransformation, imuNow);
            std::memcpy(lastImuTransformation, imuNow, sizeof(imuNow));
        }
    }
    // tf pieces
    struct Q { double x, y, z, w; };
    static Q setRPY(double roll, double pitch, double yaw) {
        double hy = yaw * 0.5, hp = pitch * 0.5, hr = roll * 0.5;
        double cy = std::cos(hy), sy = std::sin(hy), cp = std::cos(hp), sp = std::sin(hp), cr = std::cos(hr), sr = std::sin(hr);
        Q q; q.x = sr * cp * cy - cr * sp * sy; q.y = cr * sp * cy + sr * cp * sy; q.z = cr * cp * sy - sr * sp * cy; q.w = cr * cp * cy + sr * sp * sy;
        return q;
    }
    static double dot(const Q& a, const Q& b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; }
    static Q slerp(const Q& a, const Q& b, double t) {
        double s = std::sqrt(dot(a, a) * dot(b, b)), dab = dot(a, b);
        double shortest = dab < 0 ? std::acos(-dab / s) * 2.0 : std::acos(dab / s) * 2.0;
        double theta = shortest / 2.0;
        if (theta == 0.0) return a;
        double d = 1.0 / std::sin(theta), s0 = std::sin((1.0 - t) * theta), s1 = std::sin(t * theta);
        double sg = dab < 0 ? -1.0 : 1.0;
        Q r; r.x = (a.x * s0 + sg * b.x * s1) * d; r.y = (a.y * s0 + sg * b.y * s1) * d; r.z = (a.z * s0 + sg * b.z * s1) * d; r.w = (a.w * s0 + sg * b.w * s1) * d;
        return r;
    }
    static void getRPY(const Q& q, double& roll, double& pitch, double& yaw) {
        double s = 2.0 / dot(q, q);
        double xs = q.x * s, ys = q.y * s, zs = q.z * s, wx = q.w * xs, wy = q.w * ys, wz = q.w * zs;
        double xx = q.x * xs, xy = q.x * ys, xz = q.x * zs, yy = q.y * ys, yz = q.y * zs, zz = q.z * zs;
        double r0x = 1.0 - (yy + zz), r1x = xy + wz, r2x = xz - wy, r2y = yz + wx, r2z = 1.0 - (xx + yy);
        if (std::fabs(r2x) >= 1) { yaw = 0; roll = std::atan2(r2y, r2z); pitch = r2x < 0 ? M_PI / 2.0 : -M_PI / 2.0; return; }
        pitch = -std::asin(r2x);
        double c = std::cos(pitch);
        roll = std::atan2(r2y / c, r2z / c); yaw = std::atan2(r1x / c, r0x / c);
    }
    void transformUpdate(const GuessCloudInfo& ci, int imuType, float imuRPYWeight, float rotation_tollerance, float z_tollerance) {
        if (ci.imuAvailable && imuType && std::abs(ci.imuPitchInit) < 1.4) {
            double w = imuRPYWeight, r, p, y;
            getRPY(slerp(setRPY(transformTobeMapped[0], 0, 0), setRPY(ci.imuRollInit, 0, 0), w), r, p, y); transformTobeMapped[0] = (float)r;
            getRPY(slerp(setRPY(0, transformTobeMapped[1], 0), setRPY(0, ci.imuPitchInit, 0), w), r, p, y); transformTobeMapped[1] = (float)p;
        }
        auto clampf = [](float v, float lim) { return v < -lim ? -lim : (v > lim ? lim : v); };
        transformTobeMapped[0] = clampf(transformTobeMapped[0], rotation_tollerance);
        transformTobeMapped[1] = clampf(transformTobeMapped[1], rotation_tollerance);
        transformTobeMapped[5] = clampf(transformTobeMapped[5], z_tollerance);
    }
};

// deskew_enabled == 0 reproduces `deskewFlag == -1 || imuAvailable == false` passthrough (:538).
inline int project_point_cloud(const PRaw* in, int n, const DeskewParams& P, double timeScanCur, const double* imuTime,
                               const double* rx, const double* ry, const double* rz, int imuPointerCur, int deskew_enabled,
                               std::vector<P4>& out, std::vector<int>* kept_index = nullptr) {
    out.clear(); if (kept_index) kept_index->clear();
    bool firstPointFlag = true; float startInv[12];
    for (int i = 0; i < n; ++i) {
        P4 p{in[i].x, in[i].y, in[i].z, in[i].i};
        float range = std::sqrt(p.x * p.x + p.y * p.y + p.z * p.z);                 // lib/common_lib.cpp:27-31
        if (range < P.lidarMinRange || range > P.lidarMaxRange) continue;           // :581
        int rowIdn = in[i].ring;
        if (rowIdn < 0 || rowIdn >= P.N_SCAN) continue;                             // :585
        if (rowIdn % P.downsampleRate != 0) continue;                               // :588
        if (i % P.point_filter_num != 0) continue;                                  // :591
        if (deskew_enabled) {                                                       // deskewPoint :536-566
            double pointTime = timeScanCur + (double)in[i].time;
            float rxc, ryc, rzc; find_rotation(pointTime, imuTime, rx, ry, rz, imuPointerCur, &rxc, &ryc, &rzc);
            float tf[12]; get_transformation(0.f, 0.f, 0.f, rxc, ryc, rzc, tf);
            if (firstPointFlag) { affine_inverse(tf, startInv); firstPointFlag = false; }
            float bt[12]; affine_mul(startInv, tf, bt);
            p = apply_affine(bt, p);
        }
        out.push_back(p); if (kept_index) kept_index->push_back(i);
    }
    return (int)out.size();
}

// ------------------------------------------------------------------------------------------------
// S — ScanContext (include/Scancontext.cpp), sequential fp64 reductions.
// desc is 20x60 ROW-major here: desc[ring*60 + sector].
// ------------------------------------------------------------------------------------------------
constexpr int SC_RING = 20, SC_SECTOR = 60; constexpr double SC_MAX_RADIUS = 80.0, SC_LIDAR_HEIGHT = 2.0;
constexpr int SC_EXCLUDE_RECENT = 30, SC_NUM_CAND = 3, SC_TREE_PERIOD = 10; constexpr double SC_SEARCH_RATIO = 0.1, SC_DIST_THRES = 0.3;

inline float xy2theta(float x, float y) {                                      // :23-36, atan on the float quotient promoted to double
    if ((x >= 0) & (y >= 0)) return (float)((180 / M_PI) * std::atan((double)(y / x)));
    if ((x < 0) & (y >= 0)) return (float)(180 - ((180 / M_PI) * std::atan((double)(y / (-x)))));
    if ((x < 0) & (y < 0)) return (float)(180 + ((180 / M_PI) * std::atan((double)(y / x))));
    return (float)(360 - ((180 / M_PI) * std::atan((double)((-y) / x))));
}

inline void make_scancontext(const P4* pts, int n, double desc[SC_RING * SC_SECTOR]) {   // :151-195
    const double NO_POINT = -1000;
    for (int k = 0; k < SC_RING * SC_SECTOR; ++k) desc[k] = NO_POINT;
    for (int k = 0; k < n; ++k) {
        float x = pts[k].x, y = pts[k].y, z = (float)(pts[k].z + SC_LIDAR_HEIGHT);
        float azim_range = std::sqrt(x * x + y * y);
        float azim_angle = xy2theta(x, y);
        if (azim_range > SC_MAX_RADIUS) continue;
        int ring_idx = std::max(std::min(SC_RING, (int)std::ceil((azim_range / SC_MAX_RADIUS) * SC_RING)), 1);
        int sctor_idx = std::max(std::min(SC_SECTOR, (int)std::ceil((azim_angle / 360.0) * SC_SECTOR)), 1);
        double& d = desc[(ring_idx - 1) * SC_SECTOR + (sctor_idx - 1)];
        if (d < z) d = z;
    }
    for (int k = 0; k < SC_RING * SC_SECTOR; ++k) if (desc[k] == NO_POINT) desc[k] = 0;
}
inline void make_ringkey(const double* desc, double rk[SC_RING]) {              // :198-211 row means
    for (int r = 0; r < SC_RING; ++r) { double s = 0; for (int c = 0; c < SC_SECTOR; ++c) s += desc[r * SC_SECTOR + c]; rk[r] = s / SC_SECTOR; }
}
inline void make_sectorkey(const double* desc, double sk[SC_SECTOR]) {          // :214-227 column means
    for (int c = 0; c < SC_SECTOR; ++c) { double s = 0; for (int r = 0; r < SC_RING; ++r) s += desc[r * SC_SECTOR + c]; sk[c] = s / SC_RING; }
}
inline int fast_align_vkey(const double* v1, const double* v2) {                // :93-113 ; circshift :39-59
    int argmin = 0; double mn = 10000000;
    for (int s = 0; s < SC_SECTOR; ++s) {
        double ss = 0;
        for (int c = 0; c < SC_SECTOR; ++c) {             // shifted[(c0+s)%60] = v2[c0]  ⇒ shifted[c] = v2[(c-s+60)%60]
            double d = v1[c] - v2[(c - s + SC_SECTOR) % SC_SECTOR]; ss += d * d;
        }
        double nrm = std::sqrt(ss);
        if (nrm < mn) { argmin = s; mn = nrm; }
    }
    return argmin;
}
inline double dist_direct_sc(const double* sc1, const double* sc2, int shift) { // :69-90 with sc2 column-shifted by `shift`
    int num_eff = 0; double sum_sim = 0;
    for (int c = 0; c < SC_SECTOR; ++c) {
        int c2 = (c - shift + SC_SECTOR) % SC_SECTOR;
        double n1 = 0, n2 = 0, dot = 0;
        for (int r = 0; r < SC_RING; ++r) { double a = sc1[r * SC_SECTOR + c], b = sc2[r * SC_SECTOR + c2]; n1 += a * a; n2 += b * b; dot += a * b; }
        n1 = std::sqrt(n1); n2 = std::sqrt(n2);
        if ((n1 == 0) | (n2 == 0)) continue;
        sum_sim = sum_sim + dot / (n1 * n2);
        num_eff = num_eff + 1;
    }
    return 1.0 - sum_sim / num_eff;               // num_eff == 0 ⇒ 0/0 = NaN, never < min
}
inline std::pair<double, int> distance_btn_scancontext(const double* sc1, const double* sc2) {   // :116-148
    double vk1[SC_SECTOR], vk2[SC_SECTOR]; make_sectorkey(sc1, vk1); make_sectorkey(sc2, vk2);
    int a = fast_align_vkey(vk1, vk2);
    const int SEARCH_RADIUS = (int)std::round(0.5 * SC_SEARCH_RATIO * SC_SECTOR);
    std::vector<int> space{a};
    for (int ii = 1; ii < SEARCH_RADIUS + 1; ++ii) { space.push_back((a + ii + SC_SECTOR) % SC_SECTOR); space.push_back((a - ii + SC_SECTOR) % SC_SECTOR); }
    std::sort(space.begin(), space.end());
    int argmin = 0; double mn = 10000000;
    for (int s : space) { double d = dist_direct_sc(sc1, sc2, s); if (d < mn) { argmin = s; mn = d; } }
    return {mn, argmin};
}
// nanoflann L2_Adaptor::evalMetric op order (include/nanoflann.hpp:383-408), dim 20, fp32
inline float ringkey_dist(const float* a, const float* b) {
    float result = 0.f;
    for (int g = 0; g < 5; ++g) {
        float d0 = a[4 * g] - b[4 * g], d1 = a[4 * g + 1] - b[4 * g + 1], d2 = a[4 * g + 2] - b[4 * g + 2], d3 = a[4 * g + 3] - b[4 * g + 3];
        result += d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
    }
    return result;
}
// exact top-3 over keys[0:ntree) by (distance, index); slots zero-initialised like the reference's vectors (:289-290)
inline void ringkey_top3(const float* keys, int ntree, const float* q, int idx[3], float d[3]) {
    int cnt = 0; for (int j = 0; j < 3; ++j) { idx[j] = 0; d[j] = 0.f; }
    float bd[3] = {INFINITY, INFINITY, INFINITY}; int bi[3] = {0, 0, 0};
    for (int k = 0; k < ntree; ++k) {
        float dist = ringkey_dist(q, keys + 20 * (size_t)k);
        if (cnt == 3 && !(dist < bd[2])) continue;
        int j = cnt < 3 ? cnt : 2;
        while (j > 0 && bd[j - 1] > dist) { bd[j] = bd[j - 1]; bi[j] = bi[j - 1]; --j; }
        bd[j] = dist; bi[j] = k; if (cnt < 3) ++cnt;
    }
    if (cnt < 3) d[2] = (std::numeric_limits<float>::max)();     // KNNResultSet::init leaves dists[capacity-1] = max (nanoflann.hpp:160-164)
    for (int j = 0; j < cnt; ++j) { idx[j] = bi[j]; d[j] = bd[j]; }
}

struct SCManager {                                    // include/Scancontext.h:60-110 data members
    std::vector<std::vector<double>> polarcontexts_;           // 1200 doubles each (row-major)
    std::vector<std::vector<float>> invkeys_mat_;              // ring key as fp32 (eig2stdvec :62-66)
    std::vector<float> tree_keys_;                             // snapshot polarcontext_invkeys_to_search_ (flattened)
    int tree_n_ = 0; int tree_making_period_conter = 0;
    void makeAndSaveScancontextAndKeys(const P4* pts, int n) {   // :236-250
        std::vector<double> sc(SC_RING * SC_SECTOR); make_scancontext(pts, n, sc.data());
        double rk[SC_RING]; make_ringkey(sc.data(), rk);
        std::vector<float> key(SC_RING); for (int r = 0; r < SC_RING; ++r) key[r] = (float)rk[r];
        polarcontexts_.push_back(std::move(sc)); invkeys_mat_.push_back(std::move(key));
    }
    void saveDescriptor(const double* desc) {                    // benchmark helper: a11/a12 on a ready descriptor
        std::vector<double> sc(desc, desc + SC_RING * SC_SECTOR);
        double rk[SC_RING]; make_ringkey(sc.data(), rk);
        std::vector<float> key(SC_RING); for (int r = 0; r < SC_RING; ++r) key[r] = (float)rk[r];
        polarcontexts_.push_back(std::move(sc)); invkeys_mat_.push_back(std::move(key));
    }
    std::pair<int, float> detectLoopClosureID(double* out_min_dist = nullptr, int* cand = nullptr) {   // :253-344
        int loop_id = -1;
        if ((int)invkeys_mat_.size() < SC_EXCLUDE_RECENT + 1) return {loop_id, 0.0f};
        const std::vector<float>& curr_key = invkeys_mat_.back();
        const std::vector<double>& curr_desc = polarcontexts_.back();
        if (tree_making_period_conter % SC_TREE_PERIOD == 0) {
            tree_n_ = (int)invkeys_mat_.size() - SC_EXCLUDE_RECENT;
            tree_keys_.resize((size_t)tree_n_ * SC_RING);
            for (int k = 0; k < tree_n_; ++k) std::memcpy(&tree_keys_[(size_t)k * SC_RING], invkeys_mat_[k].data(), SC_RING * sizeof(float));
        }
        tree_making_period_conter = tree_making_period_conter + 1;
        double min_dist = 10000000; int nn_align = 0, nn_idx = 0;
        int cidx[3]; float cd[3]; ringkey_top3(tree_keys_.data(), tree_n_, curr_key.data(), cidx, cd);
        for (int c = 0; c < SC_NUM_CAND; ++c) {
            auto r = distance_btn_scancontext(curr_desc.data(), polarcontexts_[cidx[c]].data());
            if (r.first < min_dist) { min_dist = r.first; nn_align = r.second; nn_idx = cidx[c]; }
        }
        if (cand) { cand[0] = cidx[0]; cand[1] = cidx[1]; cand[2] = cidx[2]; }
        if (out_min_dist) *out_min_dist = min_dist;
        if (min_dist < SC_DIST_THRES) loop_id = nn_idx;
        float yaw_diff_rad = (float)((float)(nn_align * (360.0 / SC_SECTOR)) * M_PI / 180.0);   // deg2rad(float) :17-20
        return {loop_id, yaw_diff_rad};
    }
};

}  // namespace liorf_oracle
