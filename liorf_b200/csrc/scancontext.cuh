// scancontext.cuh — ScanContext on the GPU (include/Scancontext.cpp).
//   makeScancontext + ring/sector keys  (:151-227)  → k_sc_bins (atomicMax scatter into 20x60 bins) + k_sc_finalize
//   detectLoopClosureID stage 1         (:289-295)  → exact fp32 ring-key top-3 in nanoflann's evalMetric op order,
//                                                     brute force over the (sharded) key database, ties by (dist, idx)
//   distanceBtnScanContext              (:116-148)  → one warp per (query, candidate): 60-shift sector-key alignment,
//                                                     then 7 column-shift cosine distances; sequential fp64 sums
// Database layout in HBM (per entry): descriptor 20x60 fp64 row-major [ring][sector] (9600 B), ring key 20 fp32 (80 B),
// sector key 60 fp64 (480 B), column norms 60 fp64 (480 B).
#pragma once
#include "prims.cuh"

namespace liorf {

constexpr int SC_RING = 20, SC_SECTOR = 60, SC_DESC = SC_RING * SC_SECTOR;
constexpr double SC_MAX_RADIUS = 80.0, SC_LIDAR_HEIGHT = 2.0, SC_DIST_THRES = 0.3;
constexpr int SC_EXCLUDE_RECENT = 30, SC_TREE_PERIOD = 10, SC_NUM_CAND = 3;
constexpr int SC_SEARCH_RADIUS = 3;        // round(0.5 * SEARCH_RATIO(0.1) * 60)

__device__ __forceinline__ unsigned f2ord(float f) { unsigned u = __float_as_uint(f); return (u & 0x80000000u) ? ~u : (u | 0x80000000u); }
__device__ __forceinline__ float ord2f(unsigned u) { return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u); }

__device__ __forceinline__ float xy2theta_dev(float x, float y) {                 // :23-36
    const double k = 180.0 / M_PI;
    if ((x >= 0) & (y >= 0)) return (float)(k * atan((double)(y / x)));
    if ((x < 0) & (y >= 0)) return (float)(180 - (k * atan((double)(y / (-x)))));
    if ((x < 0) & (y < 0)) return (float)(180 + (k * atan((double)(y / x))));
    return (float)(360 - (k * atan((double)((-y) / x))));
}

// bins: 1200 ordered-uint, pre-set to f2ord(-1000.f)
__global__ void __launch_bounds__(256) k_sc_bins(const float4* __restrict__ pts, Count cnt, unsigned* __restrict__ bins) {
    __shared__ unsigned s_bins[SC_DESC];
    const unsigned init = f2ord(-1000.f);
    for (int i = threadIdx.x; i < SC_DESC; i += blockDim.x) s_bins[i] = init;
    __syncthreads();
    const int n = cnt.get();
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float4 p = pts[i];
        float z = (float)((double)p.z + SC_LIDAR_HEIGHT);                        // :168
        float azim_range = sqrtf(p.x * p.x + p.y * p.y);
        float azim_angle = xy2theta_dev(p.x, p.y);
        if ((double)azim_range > SC_MAX_RADIUS) continue;                        // :175
        int ring_idx = max(min(SC_RING, (int)ceil(((double)azim_range / SC_MAX_RADIUS) * SC_RING)), 1);
        int sctor_idx = max(min(SC_SECTOR, (int)ceil(((double)azim_angle / 360.0) * SC_SECTOR)), 1);
        atomicMax(&s_bins[(ring_idx - 1) * SC_SECTOR + (sctor_idx - 1)], f2ord(z));
    }
    __syncthreads();
    for (int i = threadIdx.x; i < SC_DESC; i += blockDim.x) if (s_bins[i] != init) atomicMax(&bins[i], s_bins[i]);
}

// One block: decode bins → descriptor (fp64), ring key (fp32), sector key, column norms; re-arms the bins.
// desc == nullptr → read the descriptor from desc_in instead of the bins (benchmark path: descriptor supplied directly).
__global__ void __launch_bounds__(64) k_sc_finalize(unsigned* __restrict__ bins, const double* __restrict__ desc_in, double* __restrict__ desc,
                                                   float* __restrict__ ringkey, double* __restrict__ sectorkey, double* __restrict__ colnorm) {
    __shared__ double s_d[SC_DESC];
    const unsigned init = f2ord(-1000.f);
    for (int i = threadIdx.x; i < SC_DESC; i += blockDim.x) {
        double v;
        if (desc_in) v = desc_in[i];
        else { float f = ord2f(bins[i]); v = (double)f; if (v == -1000.0) v = 0.0; bins[i] = init; }    // :187-190
        s_d[i] = v; desc[i] = v;
    }
    __syncthreads();
    const int t = threadIdx.x;
    if (t < SC_RING) { double s = 0; for (int c = 0; c < SC_SECTOR; ++c) s += s_d[t * SC_SECTOR + c]; ringkey[t] = (float)(s / SC_SECTOR); }   // :198-211, :62-66
    if (t < SC_SECTOR) {
        double s = 0, q = 0;
        for (int r = 0; r < SC_RING; ++r) { double v = s_d[r * SC_SECTOR + t]; s += v; q += v * v; }
        sectorkey[t] = s / SC_RING;                                               // :214-227
        colnorm[t] = sqrt(q);                                                     // VectorXd::norm() of the column (:75-81)
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Stage 1: ring-key top-3.  nanoflann L2_Adaptor::evalMetric op order (include/nanoflann.hpp:383-408).
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float ringkey_dist_dev(const float (&a)[20], const float4* __restrict__ b5 /*5 x float4*/) {
    float result = 0.f;
#pragma unroll
    for (int g = 0; g < 5; ++g) {
        float4 b = b5[g];
        float d0 = a[4 * g] - b.x, d1 = a[4 * g + 1] - b.y, d2 = a[4 * g + 2] - b.z, d3 = a[4 * g + 3] - b.w;
        result += d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
    }
    return result;
}
struct Top3 { float d[3]; int i[3]; };
__device__ __forceinline__ void top3_init(Top3& t) { for (int j = 0; j < 3; ++j) { t.d[j] = INFINITY; t.i[j] = 0x7fffffff; } }
__device__ __forceinline__ void top3_insert(Top3& t, float d, int i) {
    if (!(d < t.d[2] || (d == t.d[2] && i < t.i[2]))) return;
    t.d[2] = d; t.i[2] = i;
#pragma unroll
    for (int j = 2; j > 0; --j)
        if (t.d[j] < t.d[j - 1] || (t.d[j] == t.d[j - 1] && t.i[j] < t.i[j - 1])) {
            float td = t.d[j]; t.d[j] = t.d[j - 1]; t.d[j - 1] = td; int ti = t.i[j]; t.i[j] = t.i[j - 1]; t.i[j - 1] = ti;
        }
}

constexpr int SCK_BLOCK = 128;          // queries per block (one query per thread)
constexpr int SCK_TILE = 256;           // keys staged in shared memory per step
// grid = (ceil(Q / SCK_BLOCK), n_chunks).  Each (query, chunk) emits a local top-3 → part[(chunk * Q + q) * 3 + j].
// LIM (batched detectLoopClosureID): query q counts key k only if k < lim[q] (k before idx_offset), the stale tree's key prefix.  The
// shared-memory staging stays block-uniform up to the largest limit of the block, so a chunk past every limit of its block stops at once.
template <bool LIM>
__global__ void __launch_bounds__(SCK_BLOCK) k_sc_knn_tile(const float* __restrict__ keys, int n_keys, int idx_offset, const float* __restrict__ qkeys, int Q,
                                                          int keys_per_chunk, float* __restrict__ part_d, int* __restrict__ part_i, const int* __restrict__ lim) {
    __shared__ float4 s_keys[SCK_TILE * 5];
    const int q = blockIdx.x * SCK_BLOCK + threadIdx.x;
    float a[20];
#pragma unroll
    for (int k = 0; k < 20; ++k) a[k] = q < Q ? __ldg(qkeys + 20 * (size_t)q + k) : 0.f;
    Top3 t; top3_init(t);
    const int k_begin = blockIdx.y * keys_per_chunk;
    int k_end = min(n_keys, k_begin + keys_per_chunk);
    int my_lim = n_keys;
    if constexpr (LIM) {
        __shared__ int s_lmax;
        my_lim = q < Q ? __ldg(lim + q) : 0;
        if (threadIdx.x == 0) s_lmax = 0;
        __syncthreads();
        atomicMax(&s_lmax, my_lim);
        __syncthreads();
        k_end = min(k_end, s_lmax);
    }
    for (int base = k_begin; base < k_end; base += SCK_TILE) {
        const int cnt = min(SCK_TILE, k_end - base);
        __syncthreads();
        const float4* src = reinterpret_cast<const float4*>(keys + 20 * (size_t)base);
        for (int i = threadIdx.x; i < cnt * 5; i += SCK_BLOCK) s_keys[i] = __ldg(src + i);
        __syncthreads();
        for (int k = 0; k < cnt; ++k) {
            float d = ringkey_dist_dev(a, s_keys + 5 * k);
            if (!LIM || base + k < my_lim) top3_insert(t, d, idx_offset + base + k);
        }
    }
    if (q < Q) {
        const size_t o = ((size_t)blockIdx.y * Q + q) * 3;
#pragma unroll
        for (int j = 0; j < 3; ++j) { part_d[o + j] = t.d[j]; part_i[o + j] = t.i[j]; }
    }
}
// merges n_parts partial top-3 lists per query by (dist, idx); part p starts at p * part_stride elements ([part][Q][3] when
// part_stride = 3 Q; the packed all-gather layout [part]{dist[Q][3], idx[Q][3]} uses 6 Q)
__global__ void __launch_bounds__(128) k_sc_merge_top3(const float* __restrict__ part_d, const int* __restrict__ part_i, int n_parts, size_t part_stride, int Q,
                                                      float* __restrict__ out_d, int* __restrict__ out_i) {
    int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= Q) return;
    Top3 t; top3_init(t);
    for (int p = 0; p < n_parts; ++p) {
        const size_t o = (size_t)p * part_stride + (size_t)q * 3;
#pragma unroll
        for (int j = 0; j < 3; ++j) { int i = part_i[o + j]; if (i != 0x7fffffff) top3_insert(t, part_d[o + j], i); }
    }
#pragma unroll
    for (int j = 0; j < 3; ++j) { out_d[3 * (size_t)q + j] = t.d[j]; out_i[3 * (size_t)q + j] = t.i[j]; }
}

// ---------------------------------------------------------------------------------------------------------------
// Stage 2: distanceBtnScanContext for (query, candidate) pairs; one warp per pair.
// cand index is GLOBAL; this rank owns [own_begin, own_begin + own_count).  Pairs it does not own are skipped
// (out left untouched → caller pre-fills +inf / -1).  cand == INT_MAX (no candidate) → dist = +inf.
// ---------------------------------------------------------------------------------------------------------------
constexpr int SCD_WARPS = 4;
__global__ void __launch_bounds__(SCD_WARPS * 32) k_sc_distance(const double* __restrict__ qdesc, const double* __restrict__ qsk, const double* __restrict__ qcn,
                                                               const int* __restrict__ cand, int n_pairs, int cand_per_query,
                                                               const double* __restrict__ db_desc, const double* __restrict__ db_sk, const double* __restrict__ db_cn,
                                                               int own_begin, int own_count, double* __restrict__ out_dist, int* __restrict__ out_shift) {
    __shared__ double s_vk1[SCD_WARPS][SC_SECTOR], s_vk2[SCD_WARPS][SC_SECTOR];
    __shared__ double s_sim[SCD_WARPS][7][SC_SECTOR];       // per fine shift: cosine of each column, NaN-free sentinel -2 = skipped
    const int w = warp_id(), l = lane_id();
    const int pair = blockIdx.x * SCD_WARPS + w;
    if (pair >= n_pairs) return;
    const int q = pair / cand_per_query;
    const int c = cand[pair];
    if (c == 0x7fffffff || c < 0) { if (l == 0) { out_dist[pair] = INFINITY; out_shift[pair] = 0; } return; }
    const int lc = c - own_begin;
    if (lc < 0 || lc >= own_count) return;
    const double* sc1 = qdesc + (size_t)q * SC_DESC; const double* sc2 = db_desc + (size_t)lc * SC_DESC;
    const double* cn1 = qcn + (size_t)q * SC_SECTOR; const double* cn2 = db_cn + (size_t)lc * SC_SECTOR;
    for (int k = l; k < SC_SECTOR; k += 32) { s_vk1[w][k] = qsk[(size_t)q * SC_SECTOR + k]; s_vk2[w][k] = db_sk[(size_t)lc * SC_SECTOR + k]; }
    __syncwarp();
    // fastAlignUsingVkey (:93-113): lane ↔ shift, sequential sum over columns; first strict minimum of the norm
    double best = 10000000.0; int best_s = 0x7fffffff;
    {   // shifts l and l + 32 of this lane as two independent sequential sums (same per-shift order, twice the ILP)
        const int sA = l, sB = l + 32;
        const bool hasB = sB < SC_SECTOR;
        double ssA = 0, ssB = 0;
        for (int k = 0; k < SC_SECTOR; ++k) {
            int kA = k - sA; if (kA < 0) kA += SC_SECTOR;
            int kB = k - (hasB ? sB : 0); if (kB < 0) kB += SC_SECTOR;
            const double v1 = s_vk1[w][k];
            const double dA = v1 - s_vk2[w][kA], dB = v1 - s_vk2[w][kB];
            ssA += dA * dA; ssB += dB * dB;
        }
        const double nA = sqrt(ssA), nB = sqrt(ssB);
        if (nA < best) { best = nA; best_s = sA; }              // ascending s within the lane ⇒ first minimum kept
        if (hasB && nB < best) { best = nB; best_s = sB; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double ob = __shfl_xor_sync(FULL, best, o); int os = __shfl_xor_sync(FULL, best_s, o);
        if (ob < best || (ob == best && os < best_s)) { best = ob; best_s = os; }
    }
    const int align = best_s == 0x7fffffff ? 0 : best_s;        // every norm >= 1e7 or NaN ⇒ argmin stays 0 (:95)
    // fine search (:123-144): shifts {align-3..align+3} mod 60, visited in ascending order
    int shifts[7];
#pragma unroll
    for (int j = 0; j < 7; ++j) shifts[j] = (align + j - SC_SEARCH_RADIUS + SC_SECTOR) % SC_SECTOR;
#pragma unroll
    for (int a = 1; a < 7; ++a) { int v = shifts[a]; int b = a - 1; while (b >= 0 && shifts[b] > v) { shifts[b + 1] = shifts[b]; --b; } shifts[b + 1] = v; }
    // lane ↔ column: dot over the 20 rings for each of the 7 shifts
    for (int k = l; k < SC_SECTOR; k += 32) {
        double a1[SC_RING];
#pragma unroll
        for (int r = 0; r < SC_RING; ++r) a1[r] = sc1[r * SC_SECTOR + k];
        const double n1 = cn1[k];
#pragma unroll
        for (int j = 0; j < 7; ++j) {
            int k2 = k - shifts[j]; if (k2 < 0) k2 += SC_SECTOR;
            const double n2 = cn2[k2];
            double dot = 0;
#pragma unroll
            for (int r = 0; r < SC_RING; ++r) dot += a1[r] * sc2[r * SC_SECTOR + k2];
            s_sim[w][j][k] = ((n1 == 0) | (n2 == 0)) ? -2.0 : dot / (n1 * n2);      // distDirectSC :73-88
        }
    }
    __syncwarp();
    // lane j < 7: sequential sum over columns for shift j
    double dist = INFINITY; int sh = 0;
    if (l < 7) {
        double sum = 0; int eff = 0;
        for (int k = 0; k < SC_SECTOR; ++k) { double v = s_sim[w][l][k]; if (v != -2.0) { sum = sum + v; eff = eff + 1; } }
        dist = 1.0 - sum / eff;                                  // eff == 0 ⇒ NaN, never selected
        sh = shifts[0];
#pragma unroll
        for (int j = 1; j < 7; ++j) if (l == j) sh = shifts[j];
    }
    // first strict minimum in ascending shift order (lane order == ascending shift)
    double mn = 10000000.0; int arg = 0;
#pragma unroll
    for (int j = 0; j < 7; ++j) {
        double dj = __shfl_sync(FULL, dist, j); int sj = __shfl_sync(FULL, sh, j);
        if (dj < mn) { mn = dj; arg = sj; }
    }
    if (l == 0) { out_dist[pair] = mn; out_shift[pair] = arg; }
}

// sharded stage 2: every (query, candidate) pair was evaluated by exactly one rank (the owner of the candidate), all others
// left +inf / 0.  gathered[part] = { double dist[3 Q]; int shift[3 Q]; } at part * stride_bytes.  Picks the owner's entry.
__global__ void __launch_bounds__(128) k_sc_combine_pairs(const unsigned char* __restrict__ gathered, int n_parts, size_t stride_bytes, int n_pairs,
                                                         double* __restrict__ out_dist, int* __restrict__ out_shift) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pairs) return;
    double d = INFINITY; int sh = 0;
    for (int p = 0; p < n_parts; ++p) {
        const double dp = reinterpret_cast<const double*>(gathered + (size_t)p * stride_bytes)[i];
        if (dp != INFINITY) { d = dp; sh = reinterpret_cast<const int*>(gathered + (size_t)p * stride_bytes + (size_t)n_pairs * 8)[i]; break; }   // NaN != inf: an owner's NaN is kept
    }
    out_dist[i] = d; out_shift[i] = sh;
}

// final decision per query (:302-340): candidates in kNN order, strict <, threshold
__global__ void __launch_bounds__(128) k_sc_decide(const double* __restrict__ pair_dist, const int* __restrict__ pair_shift, const int* __restrict__ cand, int Q,
                                                  int* __restrict__ loop_id, int* __restrict__ shift, double* __restrict__ dist) {
    int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= Q) return;
    double mn = 10000000.0; int al = 0, nn = 0;
#pragma unroll
    for (int c = 0; c < SC_NUM_CAND; ++c) { double d = pair_dist[3 * (size_t)q + c]; if (d < mn) { mn = d; al = pair_shift[3 * (size_t)q + c]; nn = cand[3 * (size_t)q + c]; } }
    loop_id[q] = mn < SC_DIST_THRES ? nn : -1; shift[q] = al; dist[q] = mn;
}

// batched detectLoopClosureID: the stored descriptor and stored ring key of database row rows1[q] - 1 (the newest row when the database
// held rows1[q] entries) → contiguous query q.  One block per query.
__global__ void __launch_bounds__(128) k_sc_gather_queries(const double* __restrict__ db_desc, const float* __restrict__ db_keys, const int* __restrict__ rows1, int Q,
                                                          double* __restrict__ qdesc, float* __restrict__ qkeys) {
    const int q = blockIdx.x; if (q >= Q) return;
    const size_t r = (size_t)(rows1[q] - 1);
    const double2* src = reinterpret_cast<const double2*>(db_desc + r * SC_DESC);
    double2* dst = reinterpret_cast<double2*>(qdesc + (size_t)q * SC_DESC);
    for (int i = threadIdx.x; i < SC_DESC / 2; i += blockDim.x) dst[i] = __ldg(src + i);
    if (threadIdx.x < SC_RING) qkeys[(size_t)q * SC_RING + threadIdx.x] = __ldg(db_keys + r * SC_RING + threadIdx.x);
}
// an unfilled kNN slot (a tree of fewer than 3 keys) is candidate 0: the reference's result vectors are zero-initialised (:289-290)
__global__ void __launch_bounds__(128) k_sc_cand_unfilled_to_zero(int* __restrict__ cand, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && cand[i] == 0x7fffffff) cand[i] = 0;
}

// keys (fp32 ring key, sector key, column norms) for externally supplied descriptors — batch version of k_sc_finalize
// batch (nullable): the sharded search's batch number, bumped once per launch (sc_shard.cuh: this is the first kernel of a batch)
__global__ void __launch_bounds__(64) k_sc_keys_batch(const double* __restrict__ desc, int n, float* __restrict__ ringkey, double* __restrict__ sectorkey,
                                                     double* __restrict__ colnorm, unsigned* batch = nullptr) {
    __shared__ double s_d[SC_DESC];
    if (batch && blockIdx.x == 0 && threadIdx.x == 0) *batch += 1u;
    const int e = blockIdx.x; if (e >= n) return;
    for (int i = threadIdx.x; i < SC_DESC; i += blockDim.x) s_d[i] = desc[(size_t)e * SC_DESC + i];
    __syncthreads();
    const int t = threadIdx.x;
    if (t < SC_RING && ringkey) { double s = 0; for (int c = 0; c < SC_SECTOR; ++c) s += s_d[t * SC_SECTOR + c]; ringkey[(size_t)e * SC_RING + t] = (float)(s / SC_SECTOR); }
    if (t < SC_SECTOR && sectorkey) {
        double s = 0, q = 0;
        for (int r = 0; r < SC_RING; ++r) { double v = s_d[r * SC_SECTOR + t]; s += v; q += v * v; }
        sectorkey[(size_t)e * SC_SECTOR + t] = s / SC_RING;
        if (colnorm) colnorm[(size_t)e * SC_SECTOR + t] = sqrt(q);
    }
}


// Ring keys only (query batches: the sector keys / column norms of a query are derived inside stage 2): ONE WARP per descriptor, lane r
// sums ring r — its 60 sectors are 480 contiguous bytes, fetched as thirty 16-byte loads that are all in flight before the first add —
// sequentially in sector order (makeRingkeyFromScancontext :214-227, the same fp64 sums as k_sc_keys_batch).  No shared memory, no barrier:
// the kernel streams the descriptors at HBM speed (9 600 B per query) instead of paying a load → barrier → 60-add chain per 64-thread CTA.
// batch (nullable): the sharded search's batch number, bumped once per launch.
constexpr int SCK_WARPS = 4;
__global__ void __launch_bounds__(32 * SCK_WARPS) k_sc_ringkeys_batch(const double* __restrict__ desc, int n, float* __restrict__ ringkey, unsigned* batch = nullptr) {
    if (batch && blockIdx.x == 0 && threadIdx.x == 0) *batch += 1u;
    const int e = blockIdx.x * SCK_WARPS + (threadIdx.x >> 5), r = threadIdx.x & 31;
    if (e >= n || r >= SC_RING) return;
    const double2* row = reinterpret_cast<const double2*>(desc + (size_t)e * SC_DESC + (size_t)r * SC_SECTOR);
    double2 v[SC_SECTOR / 2];
#pragma unroll
    for (int c = 0; c < SC_SECTOR / 2; ++c) v[c] = __ldg(row + c);
    double s = 0;
#pragma unroll
    for (int c = 0; c < SC_SECTOR / 2; ++c) { s += v[c].x; s += v[c].y; }
    ringkey[(size_t)e * SC_RING + r] = (float)(s / SC_SECTOR);
}

}  // namespace liorf
