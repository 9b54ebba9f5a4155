// voxelgrid.cuh — pcl::VoxelGrid<PointXYZI> leaf-centroid downsample on the GPU.
// Replaces the filter behind downsampleCurrentScan (src/mapOptmization.cpp:1061-1067) and
// downSizeFilterLocalMapSurf in extractCloud (src/mapOptmization.cpp:1037-1038).
//
// Pipeline (all counts stay on the device):
//   k_vg_minmax   : componentwise min/max, last block derives min_b / div_b / multipliers and PCL's overflow guard
//   k_vg_keys     : int voxel index per point (bit-exact with PCL's float floor arithmetic)
//   radix sort    : stable (key, point index) sort — 4 x 8-bit passes
//   scan          : segment heads → output slot; segment start table
//   k_vg_centroid : one thread per voxel; sequential fp32 sums in ascending input index, divided by (float)count
// HBM traffic (algorithmic): 16 N in + 16 N_out out; the sort moves 8 N per pass on top (L2 resident for one scan).
#pragma once
#include <cstdlib>
#include "prims.cuh"

namespace liorf {

struct VoxMeta {
    float minp[3], maxp[3];
    int min_b[3], div_b[3];
    int mul1, mul2;
    float inv;
    int overflow;     // PCL: "Leaf size is too small for the input dataset" → output = input
    int n;
};

struct VoxelGridWork {
    DevBuf<float> partial;          // per-block min/max (6 floats each)
    DevBuf<unsigned> keys;
    DevBuf<unsigned> seg_start;     // start of each voxel segment in the sorted order (+ sentinel)
    DevMem<VoxMeta> meta;
    int* mm_counter = nullptr;      // view: a zero-initialised word of the context's counters
    SortWork sort;
    ScanWork scan;
    bool small_attr_set = false;
    bool force_large = false;       // tests: run the multi-kernel path on small clouds too
    // one-kernel path (k_vg_fused)
    DevBuf<float4> pts_sorted; DevBuf<unsigned> cta_hist; DevBuf<unsigned> cta_heads;
    DevMem<unsigned> fused_bar;     // [2], zero-initialised once
    int* err_flag = nullptr;        // view: the context's error flag
    bool force_multi = false;       // tests: never take the one-kernel path
    DevMem<unsigned long long> dbg;      // debug: phase stamps of the one-kernel path
    int last_launches = 0;          // kernels (and memsets) the last voxel_grid_device call enqueued
};

constexpr int VG_MM_BLOCK = 256;

__global__ void __launch_bounds__(VG_MM_BLOCK) k_vg_minmax(const float4* __restrict__ pts, Count cnt, float leaf, float* __restrict__ partial,
                                                           int* counter, VoxMeta* __restrict__ meta) {
    const int n = cnt.get();
    float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float4 p = pts[i];
        mn[0] = fminf(mn[0], p.x); mx[0] = fmaxf(mx[0], p.x);
        mn[1] = fminf(mn[1], p.y); mx[1] = fmaxf(mx[1], p.y);
        mn[2] = fminf(mn[2], p.z); mx[2] = fmaxf(mx[2], p.z);
    }
    __shared__ float s_red[VG_MM_BLOCK / 32][6];
    __shared__ bool s_last;
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { mn[a] = fminf(mn[a], __shfl_xor_sync(FULL, mn[a], o)); mx[a] = fmaxf(mx[a], __shfl_xor_sync(FULL, mx[a], o)); }
    if (lane_id() == 0) { for (int a = 0; a < 3; ++a) { s_red[warp_id()][a] = mn[a]; s_red[warp_id()][3 + a] = mx[a]; } }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < VG_MM_BLOCK / 32; ++w) for (int a = 0; a < 3; ++a) { mn[a] = fminf(mn[a], s_red[w][a]); mx[a] = fmaxf(mx[a], s_red[w][3 + a]); }
        for (int a = 0; a < 3; ++a) { partial[blockIdx.x * 6 + a] = mn[a]; partial[blockIdx.x * 6 + 3 + a] = mx[a]; }
        __threadfence();
        int t = atomicAdd(counter, 1);
        s_last = (t == (int)gridDim.x - 1);
    }
    __syncthreads();
    if (!s_last) return;
    if (threadIdx.x < 32) {                      // last block: warp 0 folds the per-block partials (min/max are order independent)
        __threadfence();
        for (int a = 0; a < 3; ++a) { mn[a] = INFINITY; mx[a] = -INFINITY; }
        for (int b = threadIdx.x; b < (int)gridDim.x; b += 32)
            for (int a = 0; a < 3; ++a) { mn[a] = fminf(mn[a], __ldcg(partial + b * 6 + a)); mx[a] = fmaxf(mx[a], __ldcg(partial + b * 6 + 3 + a)); }
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { mn[a] = fminf(mn[a], __shfl_xor_sync(FULL, mn[a], o)); mx[a] = fmaxf(mx[a], __shfl_xor_sync(FULL, mx[a], o)); }
    }
    if (threadIdx.x == 0) {
        *counter = 0;
        VoxMeta m;
        m.n = n;
        m.inv = 1.0f / leaf;
        if (n == 0) { for (int a = 0; a < 3; ++a) { mn[a] = 0.f; mx[a] = 0.f; } }
        long long d[3];
        for (int a = 0; a < 3; ++a) {
            m.minp[a] = mn[a]; m.maxp[a] = mx[a];
            d[a] = (long long)((mx[a] - mn[a]) * m.inv) + 1;
            m.min_b[a] = (int)floorf(mn[a] * m.inv);
            int max_b = (int)floorf(mx[a] * m.inv);
            m.div_b[a] = max_b - m.min_b[a] + 1;
        }
        m.overflow = (n > 0 && d[0] * d[1] * d[2] > 2147483647LL) ? 1 : 0;
        m.mul1 = m.div_b[0]; m.mul2 = m.div_b[0] * m.div_b[1];
        *meta = m;
    }
}

__global__ void __launch_bounds__(256) k_vg_keys(const float4* __restrict__ pts, Count cnt, const VoxMeta* __restrict__ meta,
                                                unsigned* __restrict__ keys) {
    const int n = cnt.get();
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float inv = meta->inv;
    if (meta->overflow) { keys[i] = (unsigned)i; return; }           // every point its own voxel ⇒ output == input
    float4 p = pts[i];
    int i0 = (int)(floorf(p.x * inv) - (float)meta->min_b[0]);
    int i1 = (int)(floorf(p.y * inv) - (float)meta->min_b[1]);
    int i2 = (int)(floorf(p.z * inv) - (float)meta->min_b[2]);
    keys[i] = (unsigned)(i0 + i1 * meta->mul1 + i2 * meta->mul2);
}

struct VgHeadLoad {
    const unsigned* keys;
    __device__ __forceinline__ unsigned operator()(int i) const { return (i == 0 || keys[i] != keys[i - 1]) ? 1u : 0u; }
};
struct VgHeadStore {
    unsigned* seg_start; Count cnt;
    __device__ __forceinline__ void operator()(int i, unsigned v, unsigned excl) const {
        if (v) seg_start[excl] = (unsigned)i;
        if (i == cnt.get() - 1) seg_start[excl + v] = (unsigned)(i + 1);       // sentinel
    }
};

__global__ void __launch_bounds__(128) k_vg_centroid(const float4* __restrict__ pts, const unsigned* __restrict__ sorted_idx,
                                                     const unsigned* __restrict__ seg_start, const unsigned* __restrict__ n_out,
                                                     float4* __restrict__ out, int* __restrict__ membership,
                                                     const unsigned* __restrict__ sorted_keys, int* __restrict__ out_keys) {
    const int nseg = (int)*n_out;
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nseg) return;
    unsigned b = seg_start[s], e = seg_start[s + 1];
    float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f;
    unsigned k = b;
    for (; k + 4 <= e; k += 4) {                  // gathers issued four at a time; the adds stay in ascending input index
        unsigned i0 = sorted_idx[k], i1 = sorted_idx[k + 1], i2 = sorted_idx[k + 2], i3 = sorted_idx[k + 3];
        float4 p0 = __ldg(pts + i0), p1 = __ldg(pts + i1), p2 = __ldg(pts + i2), p3 = __ldg(pts + i3);
        sx += p0.x; sy += p0.y; sz += p0.z; si += p0.w;
        sx += p1.x; sy += p1.y; sz += p1.z; si += p1.w;
        sx += p2.x; sy += p2.y; sz += p2.z; si += p2.w;
        sx += p3.x; sy += p3.y; sz += p3.z; si += p3.w;
        if (membership) { membership[i0] = s; membership[i1] = s; membership[i2] = s; membership[i3] = s; }
    }
    for (; k < e; ++k) {
        unsigned idx = sorted_idx[k];
        float4 p = __ldg(pts + idx);
        sx += p.x; sy += p.y; sz += p.z; si += p.w;
        if (membership) membership[idx] = s;
    }
    float c = (float)(e - b);
    out[s] = make_float4(sx / c, sy / c, sz / c, si / c);
    if (out_keys) out_keys[s] = (int)sorted_keys[b];
}

// ---------------------------------------------------------------------------------------------------------------
// Tiny clouds (<= 3072 points: Livox scans after point_filter_num, key-pose clouds, test fixtures): the whole filter in ONE
// launch by ONE CTA instead of nine dependent launches (22 us instead of 61 us at 3000 points).  Measured on B200 the
// single CTA stops paying at ~10 k points — one SM cannot issue the sort's instructions fast enough — so larger clouds
// keep the multi-kernel radix path.
//   min/max → keys → stable LSD radix sort of (key, input index) in shared memory (4-bit digits, 4 items per thread held in
//   registers in blocked order, ranks from a block-wide scan of per-thread digit counts — only as many passes as the voxel index
//   has bits) → segment heads → exclusive scan → centroids.  Results are bit-identical to the large path.
// ---------------------------------------------------------------------------------------------------------------
constexpr int VGS_THREADS = 768;
constexpr int VGS_E = 4;                              // items per thread, held in registers in blocked order
constexpr int VGS_CAP = VGS_E * VGS_THREADS;          // 3072 points: (key u32 + index u16) x 3072 = 18 KB of shared memory
constexpr int VGS_SMEM = VGS_CAP * 6 + 16 * VGS_THREADS * 2;     // keys + indices + digit counters


// stable block-wide LSD radix sort of P = E * VGS_THREADS (key, index) pairs living in shared memory.  Items are held in
// registers in blocked order (indices packed two per register, in-thread ranks four per register).
template <int E>
__device__ __forceinline__ void vgs_radix_sort(unsigned* s_key, unsigned short* s_idx, unsigned short* s_cnt, unsigned* s_wsum, int bits) {
    const int tid = threadIdx.x;
    unsigned key[E]; unsigned ip[E / 2];
    const unsigned* s_idx2 = reinterpret_cast<const unsigned*>(s_idx);
#pragma unroll
    for (int u = 0; u < E; ++u) key[u] = s_key[tid * E + u];
#pragma unroll
    for (int u = 0; u < E / 2; ++u) ip[u] = s_idx2[tid * (E / 2) + u];
    for (int shift = 0; shift < bits; shift += 4) {
        unsigned long long lo = 0, hi = 0;                      // sixteen 8-bit counters (E <= 32 fits)
        unsigned rk[E / 4];
#pragma unroll
        for (int u = 0; u < E; ++u) {
            const unsigned d = (key[u] >> shift) & 15u;
            const unsigned sh = (d & 7u) * 8u;
            const unsigned long long sel = d < 8u ? lo : hi;
            const unsigned r = (unsigned)(sel >> sh) & 0xffu;
            if ((u & 3) == 0) rk[u / 4] = r; else rk[u / 4] |= r << (8 * (u & 3));
            const unsigned long long inc = 1ull << sh;
            lo += d < 8u ? inc : 0ull; hi += d < 8u ? 0ull : inc;
        }
#pragma unroll
        for (int d = 0; d < 16; ++d) s_cnt[d * VGS_THREADS + tid] = (unsigned short)(((d < 8 ? lo : hi) >> ((d & 7) * 8)) & 0xffu);
        __syncthreads();
        // exclusive scan over the 16 x VGS_THREADS counters in (digit, thread) order: thread t rakes entries [16 t, 16 t + 16)
        unsigned sum = 0;
#pragma unroll
        for (int k = 0; k < 16; ++k) sum += s_cnt[tid * 16 + k];
        unsigned incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned v = __shfl_up_sync(FULL, incl, o); if (lane_id() >= o) incl += v; }
        if (lane_id() == 31) s_wsum[warp_id()] = incl;
        __syncthreads();
        if (warp_id() == 0) {
            const unsigned v = lane_id() < VGS_THREADS / 32 ? s_wsum[lane_id()] : 0u; unsigned inc2 = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const unsigned w = __shfl_up_sync(FULL, inc2, o); if (lane_id() >= o) inc2 += w; }
            if (lane_id() < VGS_THREADS / 32) s_wsum[lane_id()] = inc2 - v;
        }
        __syncthreads();
        unsigned run = s_wsum[warp_id()] + incl - sum;
#pragma unroll
        for (int k = 0; k < 16; ++k) { const unsigned v = s_cnt[tid * 16 + k]; s_cnt[tid * 16 + k] = (unsigned short)run; run += v; }
        __syncthreads();
#pragma unroll
        for (int u = 0; u < E; ++u) {
            const unsigned d = (key[u] >> shift) & 15u;
            const unsigned dest = (unsigned)s_cnt[d * VGS_THREADS + tid] + ((rk[u / 4] >> (8 * (u & 3))) & 0xffu);
            s_key[dest] = key[u]; s_idx[dest] = (unsigned short)((u & 1) ? (ip[u / 2] >> 16) : (ip[u / 2] & 0xffffu));
        }
        __syncthreads();
        if (shift + 4 < bits) {
#pragma unroll
            for (int u = 0; u < E; ++u) key[u] = s_key[tid * E + u];
#pragma unroll
            for (int u = 0; u < E / 2; ++u) ip[u] = s_idx2[tid * (E / 2) + u];
        }
    }
}

__global__ void __launch_bounds__(VGS_THREADS, 1) k_vg_small(const float4* __restrict__ pts, Count cnt, float leaf, float4* __restrict__ out, int* __restrict__ n_out_dev,
                                                            int* __restrict__ membership, int* __restrict__ out_keys, VoxMeta* __restrict__ meta_out,
                                                            unsigned* __restrict__ seg_start) {
    extern __shared__ unsigned char vgs_smem[];
    unsigned* s_key = reinterpret_cast<unsigned*>(vgs_smem);
    unsigned short* s_idx = reinterpret_cast<unsigned short*>(vgs_smem + (size_t)VGS_CAP * 4);
    unsigned short* s_cnt = reinterpret_cast<unsigned short*>(vgs_smem + (size_t)VGS_CAP * 6);
    __shared__ float s_red[VGS_THREADS / 32][6];
    __shared__ VoxMeta s_meta;
    __shared__ unsigned s_wsum[32];
    __shared__ unsigned s_total;
    const int n = cnt.get();
    const int tid = threadIdx.x;
    if (n <= 0) { if (tid == 0) { *n_out_dev = 0; } return; }
    // ---- 1. bounds (min/max are order independent) ----
    float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int i = tid; i < n; i += VGS_THREADS) {
        const float4 p = pts[i];
        mn[0] = fminf(mn[0], p.x); mx[0] = fmaxf(mx[0], p.x);
        mn[1] = fminf(mn[1], p.y); mx[1] = fmaxf(mx[1], p.y);
        mn[2] = fminf(mn[2], p.z); mx[2] = fmaxf(mx[2], p.z);
    }
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { mn[a] = fminf(mn[a], __shfl_xor_sync(FULL, mn[a], o)); mx[a] = fmaxf(mx[a], __shfl_xor_sync(FULL, mx[a], o)); }
    if (lane_id() == 0) { for (int a = 0; a < 3; ++a) { s_red[warp_id()][a] = mn[a]; s_red[warp_id()][3 + a] = mx[a]; } }
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < VGS_THREADS / 32; ++w) for (int a = 0; a < 3; ++a) { mn[a] = fminf(mn[a], s_red[w][a]); mx[a] = fmaxf(mx[a], s_red[w][3 + a]); }
        VoxMeta m;
        m.n = n;
        m.inv = 1.0f / leaf;
        long long d[3];
        for (int a = 0; a < 3; ++a) {
            m.minp[a] = mn[a]; m.maxp[a] = mx[a];
            d[a] = (long long)((mx[a] - mn[a]) * m.inv) + 1;
            m.min_b[a] = (int)floorf(mn[a] * m.inv);
            const int max_b = (int)floorf(mx[a] * m.inv);
            m.div_b[a] = max_b - m.min_b[a] + 1;
        }
        m.overflow = (d[0] * d[1] * d[2] > 2147483647LL) ? 1 : 0;
        m.mul1 = m.div_b[0]; m.mul2 = m.div_b[0] * m.div_b[1];
        s_meta = m; *meta_out = m;
    }
    __syncthreads();
    // ---- 2. keys (same float arithmetic as k_vg_keys), padded to VGS_CAP items with keys that sort last ----
    const int P = VGS_CAP;
    int bits;
    {
        const float inv = s_meta.inv; const int b0 = s_meta.min_b[0], b1 = s_meta.min_b[1], b2 = s_meta.min_b[2], m1 = s_meta.mul1, m2 = s_meta.mul2;
        const bool ovf = s_meta.overflow != 0;
        // the div_b product can pass 2^32 under PCL's guard (which bounds the d product): its keys wrap and span all 32 bits
        const unsigned max_key = ovf ? (unsigned)(n - 1) : (unsigned)min((long long)s_meta.div_b[0] * s_meta.div_b[1] * s_meta.div_b[2] - 1, 0xffffffffLL);
        bits = 32 - __clz(max_key | 1u);
        for (int i = tid; i < P; i += VGS_THREADS) {
            unsigned key = 0xffffffffu;
            if (i < n) {
                if (ovf) key = (unsigned)i;                              // every point its own voxel ⇒ output == input
                else {
                    const float4 p = pts[i];
                    const int i0 = (int)(floorf(p.x * inv) - (float)b0), i1 = (int)(floorf(p.y * inv) - (float)b1), i2 = (int)(floorf(p.z * inv) - (float)b2);
                    key = (unsigned)(i0 + i1 * m1 + i2 * m2);
                }
            }
            s_key[i] = key; s_idx[i] = (unsigned short)i;
        }
    }
    __syncthreads();
    // ---- 3. stable sort by key (ties keep ascending input index; the padding ties with the largest key and stays behind it) ----
    vgs_radix_sort<VGS_E>(s_key, s_idx, s_cnt, s_wsum, bits);
    // ---- 4. segment heads → exclusive scan (thread t owns the consecutive items [t * per, (t + 1) * per)) ----
    const int per = P / VGS_THREADS;
    const int i_begin = tid * per;
    unsigned local = 0;
    for (int u = 0; u < per; ++u) { const int i = i_begin + u; if (i < n && (i == 0 || s_key[i] != s_key[i - 1])) ++local; }
    unsigned incl = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const unsigned v = __shfl_up_sync(FULL, incl, o); if (lane_id() >= o) incl += v; }
    if (lane_id() == 31) s_wsum[warp_id()] = incl;
    __syncthreads();
    if (warp_id() == 0) {
        const unsigned v = lane_id() < VGS_THREADS / 32 ? s_wsum[lane_id()] : 0u; unsigned inc2 = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned u = __shfl_up_sync(FULL, inc2, o); if (lane_id() >= o) inc2 += u; }
        if (lane_id() < VGS_THREADS / 32) s_wsum[lane_id()] = inc2 - v;  // exclusive warp offsets
        if (lane_id() == 31) s_total = inc2;
    }
    __syncthreads();
    unsigned pos = s_wsum[warp_id()] + incl - local;
    for (int u = 0; u < per; ++u) { const int i = i_begin + u; if (i < n && (i == 0 || s_key[i] != s_key[i - 1])) seg_start[pos++] = (unsigned)i; }
    const int nseg = (int)s_total;
    if (tid == 0) { seg_start[nseg] = (unsigned)n; *n_out_dev = nseg; }
    __syncthreads();
    // ---- 5. centroids: one thread per voxel, sequential fp32 sums in ascending input index, divided by (float)count ----
    for (int s = tid; s < nseg; s += VGS_THREADS) {
        const unsigned b = seg_start[s], e = seg_start[s + 1];
        float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f;
        for (unsigned k = b; k < e; ++k) {
            const unsigned idx = s_idx[k];
            const float4 p = __ldg(pts + idx);
            sx += p.x; sy += p.y; sz += p.z; si += p.w;
            if (membership) membership[idx] = s;
        }
        const float c = (float)(e - b);
        out[s] = make_float4(sx / c, sy / c, sz / c, si / c);
        if (out_keys) out_keys[s] = (int)s_key[b];
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Larger clouds (a 120 k-point scan, a 650 k-point local map): the whole filter as ONE cooperative kernel.
// The multi-kernel path below spends 93 us on a KITTI scan — ten dependent launches whose kernels are each latency-bound (a
// look-back chain over 58 tiles per radix pass, a centroid kernel that chases index → point through L2 four points at a time).
// Here the CTAs stay resident, each owns a CONTIGUOUS chunk of the points (chunk order == input order, which is what keeps the
// sort stable), and the phases are separated by a grid barrier of ~1 us:
//   bounds      block min/max → per-CTA partials | barrier | every CTA folds the partials and derives PCL's min_b / div_b itself
//   radix pass  (only as many 8-bit passes as the largest voxel index has bits: 3 for a KITTI scan at 0.4 m)
//               per-CTA digit histogram of the chunk | barrier | every CTA sums the histograms of the CTAs before it (and all of
//               them: the digit bases) — 148 x 1 KB, no look-back chain | stable scatter of the chunk, tile by tile | barrier.
//               Pass 0 computes the voxel index from the point (no key kernel); a chunk of one tile keeps keys, values and ranks
//               in registers between histogram and scatter; the LAST pass also moves the 16-byte point to its sorted place.
//   heads       per-CTA count of segment heads | barrier | segment starts written at (heads of earlier CTAs) + local rank | barrier
//   centroids   one thread per voxel over CONTIGUOUS points: sequential fp32 sums in ascending input index (the stable sort's
//               order), eight loads in flight.
// Results are bit-identical to the multi-kernel path (tests force either).  The grid is chosen by the caller: all SMs, or the few
// SMs the persistent solver leaves free when the next frame's front end runs beside it.
// ---------------------------------------------------------------------------------------------------------------
constexpr int VGF_THREADS = 512;
constexpr int VGF_WARPS = VGF_THREADS / 32;
constexpr int VGF_IPT = 2;
constexpr int VGF_TILE = VGF_THREADS * VGF_IPT;        // 1024 points per tile
constexpr int VGF_PF = 10;                             // histogram rows a thread of the prefix step keeps in flight (2 x 10 x 8 covers 148 CTAs)

struct VgFusedArgs {
    const float4* pts; Count cnt; float leaf;
    float4* out; int* n_out; int* membership; int* out_keys; VoxMeta* meta;
    unsigned* keys_a; unsigned* keys_b; unsigned* vals_a; unsigned* vals_b;      // ping-pong (key, input index)
    float4* pts_sorted; unsigned* seg_start;
    float* partial_mm;            // [grid][6]
    unsigned* cta_hist;           // [grid][RADIX]
    unsigned* cta_heads;          // [grid]
    unsigned* bar;                // [2]: arrivals, generation (zero-initialised once; reusable across launches)
    int* err_flag;
    unsigned long long* dbg;      // optional [32] %globaltimer stamps of CTA 0 at the phase boundaries (nullptr = off)
};

// grid barrier for co-resident CTAs: arrivals are counted in ONE monotonic word per launch (barrier k is complete at (k + 1) x grid);
// a CTA arrives with a fire-and-forget red.release (its threads' earlier writes are ordered before it by the CTA barrier in front) and
// polls with ld.acquire — one fence, no atomic round trip, no reset between barriers.  The last CTA to LEAVE the kernel zeroes the
// words for the next launch (vgf_finish).
__device__ __forceinline__ void vgf_grid_barrier(unsigned* bar, unsigned& gen, int* err_flag) {
    __syncthreads();
    ++gen;
    if (threadIdx.x == 0) {
        asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(bar) : "memory");
        const unsigned target = gen * gridDim.x;
        unsigned v, spins = 0;
        while (true) {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(bar) : "memory");
            if (v >= target) break;
            if (++spins > SPIN_LIMIT) { atomicExch(err_flag, 1); break; }
        }
    }
    __syncthreads();
}
__device__ __forceinline__ void vgf_finish(unsigned* bar) {
    __syncthreads();
    if (threadIdx.x == 0 && atomicAdd(bar + 1, 1u) == gridDim.x - 1) { bar[0] = 0u; bar[1] = 0u; __threadfence(); }
}

__device__ __forceinline__ unsigned vgf_key(const float4 p, float inv, int b0, int b1, int b2, int m1, int m2) {
    const int i0 = (int)(floorf(p.x * inv) - (float)b0), i1 = (int)(floorf(p.y * inv) - (float)b1), i2 = (int)(floorf(p.z * inv) - (float)b2);
    return (unsigned)(i0 + i1 * m1 + i2 * m2);
}

__global__ void __launch_bounds__(VGF_THREADS, 2) k_vg_fused(VgFusedArgs a) {
    __shared__ float s_red[VGF_WARPS][6];
    __shared__ VoxMeta s_meta;
    __shared__ unsigned s_whist[VGF_WARPS][RADIX];      // per-warp digit counts of a tile → exclusive warp offsets
    __shared__ unsigned s_hist[RADIX];                  // digit counts of the CTA's chunk
    __shared__ unsigned s_run[RADIX];                   // next output position per digit
    __shared__ unsigned s_warp[VGF_WARPS + 1];
    __shared__ uint4 s_part4[2][8][RADIX / 4];          // prefix step: (before me | all) x 8 row groups x 64 digit quads
    const int tid = threadIdx.x, w = tid >> 5, l = tid & 31;
    const int G = (int)gridDim.x, c = (int)blockIdx.x;
    const int n = a.cnt.get();
    unsigned gen = 0;                                    // barriers passed so far (every thread counts along)
    int dbg_k = 0;
    auto stamp = [&]() { if (a.dbg && c == 0 && tid == 0 && dbg_k < 32) { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); a.dbg[dbg_k] = t; } ++dbg_k; };
    stamp();
    if (n <= 0) { if (c == 0 && tid == 0) *a.n_out = 0; return; }        // (no barrier was entered: the words stay zero)
    // ---- bounds (min/max are order independent) ----
    {
        float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
        for (int i = c * VGF_THREADS + tid; i < n; i += G * VGF_THREADS) {
            const float4 p = a.pts[i];
            mn[0] = fminf(mn[0], p.x); mx[0] = fmaxf(mx[0], p.x);
            mn[1] = fminf(mn[1], p.y); mx[1] = fmaxf(mx[1], p.y);
            mn[2] = fminf(mn[2], p.z); mx[2] = fmaxf(mx[2], p.z);
        }
#pragma unroll
        for (int k = 0; k < 3; ++k)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { mn[k] = fminf(mn[k], __shfl_xor_sync(FULL, mn[k], o)); mx[k] = fmaxf(mx[k], __shfl_xor_sync(FULL, mx[k], o)); }
        if (l == 0) { for (int k = 0; k < 3; ++k) { s_red[w][k] = mn[k]; s_red[w][3 + k] = mx[k]; } }
        __syncthreads();
        if (tid < 6) {
            float v = s_red[0][tid];
            for (int ww = 1; ww < VGF_WARPS; ++ww) v = tid < 3 ? fminf(v, s_red[ww][tid]) : fmaxf(v, s_red[ww][tid]);
            __stcg(a.partial_mm + c * 6 + tid, v);
        }
        stamp();
        vgf_grid_barrier(a.bar, gen, a.err_flag);
        stamp();
        if (w == 0) {
            for (int k = 0; k < 3; ++k) { mn[k] = INFINITY; mx[k] = -INFINITY; }
            for (int b = l; b < G; b += 32)
                for (int k = 0; k < 3; ++k) { mn[k] = fminf(mn[k], __ldcg(a.partial_mm + b * 6 + k)); mx[k] = fmaxf(mx[k], __ldcg(a.partial_mm + b * 6 + 3 + k)); }
#pragma unroll
            for (int k = 0; k < 3; ++k)
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) { mn[k] = fminf(mn[k], __shfl_xor_sync(FULL, mn[k], o)); mx[k] = fmaxf(mx[k], __shfl_xor_sync(FULL, mx[k], o)); }
            if (l == 0) {
                VoxMeta m;
                m.n = n;
                m.inv = 1.0f / a.leaf;
                long long d[3];
                for (int k = 0; k < 3; ++k) {
                    m.minp[k] = mn[k]; m.maxp[k] = mx[k];
                    d[k] = (long long)((mx[k] - mn[k]) * m.inv) + 1;
                    m.min_b[k] = (int)floorf(mn[k] * m.inv);
                    const int max_b = (int)floorf(mx[k] * m.inv);
                    m.div_b[k] = max_b - m.min_b[k] + 1;
                }
                m.overflow = (d[0] * d[1] * d[2] > 2147483647LL) ? 1 : 0;
                m.mul1 = m.div_b[0]; m.mul2 = m.div_b[0] * m.div_b[1];
                s_meta = m;
                if (c == 0) *a.meta = m;
            }
        }
        __syncthreads();
    }
    const float inv = s_meta.inv; const int b0 = s_meta.min_b[0], b1 = s_meta.min_b[1], b2 = s_meta.min_b[2], m1 = s_meta.mul1, m2 = s_meta.mul2;
    if (s_meta.overflow) {
        // PCL: "Leaf size is too small for the input dataset" → output = input (every point its own voxel, key = index)
        for (int i = c * VGF_THREADS + tid; i < n; i += G * VGF_THREADS) {
            const float4 p = a.pts[i];
            float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f;
            sx += p.x; sy += p.y; sz += p.z; si += p.w;
            a.out[i] = make_float4(sx / 1.f, sy / 1.f, sz / 1.f, si / 1.f);
            if (a.membership) a.membership[i] = i;
            if (a.out_keys) a.out_keys[i] = i;
            a.seg_start[i] = (unsigned)i;
        }
        if (c == 0 && tid == 0) { a.seg_start[n] = (unsigned)n; *a.n_out = n; }
        vgf_finish(a.bar);
        return;
    }
    // the div_b product can pass 2^32 under PCL's guard (which bounds the d product): its keys wrap and span all 32 bits
    const unsigned max_key = (unsigned)min((long long)s_meta.div_b[0] * s_meta.div_b[1] * s_meta.div_b[2] - 1, 0xffffffffLL);
    const int bits = 32 - __clz(max_key | 1u);
    const int npass = (bits + RADIX_BITS - 1) / RADIX_BITS;
    // the CTA's chunk of the input order: whole tiles, contiguous
    const int chunk = (((n + G - 1) / G + VGF_TILE - 1) / VGF_TILE) * VGF_TILE;
    const int lo = min(n, c * chunk), hi = min(n, lo + chunk);
    const bool one_tile = chunk == VGF_TILE;
    const unsigned lt_mask = (1u << l) - 1u;
    unsigned* kin = a.keys_a; unsigned* kout = a.keys_b; unsigned* vin = a.vals_a; unsigned* vout = a.vals_b;
    for (int pass = 0; pass < npass; ++pass) {
        const int shift = RADIX_BITS * pass;
        const bool last = pass == npass - 1;
        unsigned key[VGF_IPT], val[VGF_IPT], rank[VGF_IPT];
        // element e of a tile is (warp, j, lane): index = tile base + w * 64 + j * 32 + l — ascending in (w, j, l)
        auto load_tile = [&](int tb) {
#pragma unroll
            for (int j = 0; j < VGF_IPT; ++j) {
                const int i = tb + w * (32 * VGF_IPT) + j * 32 + l;
                const bool valid = i < hi;
                if (pass == 0) { key[j] = valid ? vgf_key(a.pts[i], inv, b0, b1, b2, m1, m2) : 0xffffffffu; val[j] = (unsigned)i; }
                else { key[j] = valid ? __ldcg(kin + i) : 0xffffffffu; val[j] = valid ? __ldcg(vin + i) : 0u; }      // written by other CTAs in the previous pass: read behind L1
            }
        };
        // per-warp stable ranks of a loaded tile (s_whist[w] must be zero on entry); leaves the warp's digit counts in s_whist[w]
        auto rank_tile = [&](int tb) {
#pragma unroll
            for (int j = 0; j < VGF_IPT; ++j) {
                const int i = tb + w * (32 * VGF_IPT) + j * 32 + l;
                const bool valid = i < hi;
                const unsigned d = (key[j] >> shift) & (RADIX - 1);
                const unsigned vm = __ballot_sync(FULL, valid);
                const unsigned mm = __match_any_sync(FULL, d) & vm;
                unsigned old = 0;
                const int leader = __ffs(mm) - 1;
                if (valid && l == leader) { old = s_whist[w][d]; s_whist[w][d] = old + __popc(mm); }
                __syncwarp();
                old = __shfl_sync(FULL, old, leader < 0 ? 0 : leader);
                rank[j] = old + __popc(mm & lt_mask);
            }
        };
        // ---- histogram of the chunk ----
        for (int i = tid; i < VGF_WARPS * RADIX; i += VGF_THREADS) (&s_whist[0][0])[i] = 0;
        if (tid < RADIX) s_hist[tid] = 0;
        __syncthreads();
        if (one_tile) {
            load_tile(lo); rank_tile(lo);
            __syncthreads();
            if (tid < RADIX) { unsigned run = 0; for (int ww = 0; ww < VGF_WARPS; ++ww) { const unsigned v = s_whist[ww][tid]; s_whist[ww][tid] = run; run += v; } s_hist[tid] = run; }
        } else {
            for (int tb = lo; tb < hi; tb += VGF_TILE) {
                load_tile(tb);
#pragma unroll
                for (int j = 0; j < VGF_IPT; ++j) {
                    const int i = tb + w * (32 * VGF_IPT) + j * 32 + l;
                    const bool valid = i < hi;
                    const unsigned d = (key[j] >> shift) & (RADIX - 1);
                    const unsigned mm = __match_any_sync(FULL, d) & __ballot_sync(FULL, valid);
                    if (valid && l == __ffs(mm) - 1) atomicAdd(&s_hist[d], (unsigned)__popc(mm));
                }
            }
        }
        __syncthreads();
        if (tid < RADIX) __stcg(a.cta_hist + (size_t)c * RADIX + tid, s_hist[tid]);
        stamp();
        vgf_grid_barrier(a.bar, gen, a.err_flag);
        stamp();
        // ---- digit bases + what the CTAs before this one hold of each digit ----
        {   // thread (g, q): rows g, g + 8, ... of the histogram matrix, digits 4q .. 4q + 3 as one 16-byte load — all of a thread's ~19 loads in flight at once
            const int q = tid & 63, g = tid >> 6;
            uint4 pre = make_uint4(0, 0, 0, 0), tot = make_uint4(0, 0, 0, 0);
            const uint4* H = reinterpret_cast<const uint4*>(a.cta_hist);
            for (int c0 = g; c0 < G; c0 += 8 * VGF_PF) {              // VGF_PF rows per thread in flight
                uint4 v[VGF_PF];
#pragma unroll
                for (int u = 0; u < VGF_PF; ++u) { const int cc = c0 + 8 * u; v[u] = cc < G ? __ldcg(H + (size_t)cc * (RADIX / 4) + q) : make_uint4(0, 0, 0, 0); }
#pragma unroll
                for (int u = 0; u < VGF_PF; ++u) {
                    tot.x += v[u].x; tot.y += v[u].y; tot.z += v[u].z; tot.w += v[u].w;
                    if (c0 + 8 * u < c) { pre.x += v[u].x; pre.y += v[u].y; pre.z += v[u].z; pre.w += v[u].w; }
                }
            }
            s_part4[0][g][q] = pre; s_part4[1][g][q] = tot;
            __syncthreads();
            unsigned mypre = 0, mytot = 0;
            if (tid < RADIX) {
                const unsigned* P0 = reinterpret_cast<const unsigned*>(&s_part4[0][0][0]);
                const unsigned* P1 = reinterpret_cast<const unsigned*>(&s_part4[1][0][0]);
#pragma unroll
                for (int gg = 0; gg < 8; ++gg) { mypre += P0[gg * RADIX + tid]; mytot += P1[gg * RADIX + tid]; }
            }
            unsigned total;
            const unsigned goff = block_excl_scan<VGF_THREADS>(mytot, s_warp, total);      // threads 0..255 hold the digits in order, the rest add 0 behind them
            if (tid < RADIX) s_run[tid] = goff + mypre;
            __syncthreads();
        }
        stamp();
        // ---- stable scatter ----
        if (one_tile) {
#pragma unroll
            for (int j = 0; j < VGF_IPT; ++j) {
                const int i = lo + w * (32 * VGF_IPT) + j * 32 + l;
                if (i < hi) {
                    const unsigned d = (key[j] >> shift) & (RADIX - 1);
                    const unsigned pos = s_run[d] + s_whist[w][d] + rank[j];
                    kout[pos] = key[j]; vout[pos] = val[j];
                    if (last) a.pts_sorted[pos] = a.pts[val[j]];
                }
            }
        } else {
            for (int tb = lo; tb < hi; tb += VGF_TILE) {
                for (int i = tid; i < VGF_WARPS * RADIX; i += VGF_THREADS) (&s_whist[0][0])[i] = 0;
                __syncthreads();
                load_tile(tb); rank_tile(tb);
                __syncthreads();
                unsigned tile_total = 0;
                if (tid < RADIX) { unsigned run = 0; for (int ww = 0; ww < VGF_WARPS; ++ww) { const unsigned v = s_whist[ww][tid]; s_whist[ww][tid] = run; run += v; } tile_total = run; }
                __syncthreads();
#pragma unroll
                for (int j = 0; j < VGF_IPT; ++j) {
                    const int i = tb + w * (32 * VGF_IPT) + j * 32 + l;
                    if (i < hi) {
                        const unsigned d = (key[j] >> shift) & (RADIX - 1);
                        const unsigned pos = s_run[d] + s_whist[w][d] + rank[j];
                        kout[pos] = key[j]; vout[pos] = val[j];
                        if (last) a.pts_sorted[pos] = a.pts[val[j]];
                    }
                }
                __syncthreads();
                if (tid < RADIX) s_run[tid] += tile_total;
            }
        }
        stamp();
        vgf_grid_barrier(a.bar, gen, a.err_flag);
        stamp();
        { unsigned* t = kin; kin = kout; kout = t; t = vin; vin = vout; vout = t; }
    }
    // sorted (key, input index) now in kin / vin, the points in pts_sorted
    // ---- segment heads: count per chunk | barrier | every head's thread sums its segment ----
    // (item pair of thread t in a tile: tb + 2t, tb + 2t + 1 — contiguous, so the block scan numbers the heads in ascending order)
    {
        auto is_head = [&](int i) { return i < hi && (i == 0 || __ldcg(kin + i) != __ldcg(kin + i - 1)); };
        unsigned f0r = 0, f1r = 0;                         // a chunk of one tile keeps its flags across the barrier
        unsigned cnt_local = 0;
        for (int tb = lo; tb < hi; tb += VGF_TILE) {
            const int i0 = tb + tid * VGF_IPT;
            f0r = is_head(i0) ? 1u : 0u; f1r = is_head(i0 + 1) ? 1u : 0u;
            cnt_local += f0r + f1r;
        }
        unsigned total;
        (void)block_excl_scan<VGF_THREADS>(cnt_local, s_warp, total);
        if (tid == 0) __stcg(a.cta_heads + c, total);
        stamp();
        vgf_grid_barrier(a.bar, gen, a.err_flag);
        stamp();
        unsigned pre = 0, tot = 0;
        for (int cc = tid; cc < G; cc += VGF_THREADS) { const unsigned v = __ldcg(a.cta_heads + cc); tot += v; if (cc < c) pre += v; }
        unsigned t1, t2;
        (void)block_excl_scan<VGF_THREADS>(pre, s_warp, t1);
        (void)block_excl_scan<VGF_THREADS>(tot, s_warp, t2);
        unsigned slot_base = t1;
        if (c == 0 && tid == 0) { *a.n_out = (int)t2; a.seg_start[t2] = (unsigned)n; }
        for (int tb = lo; tb < hi; tb += VGF_TILE) {
            const int i0 = tb + tid * VGF_IPT;
            unsigned f[VGF_IPT];
            if (one_tile) { f[0] = f0r; f[1] = f1r; } else { f[0] = is_head(i0) ? 1u : 0u; f[1] = is_head(i0 + 1) ? 1u : 0u; }
            unsigned tile_total;
            const unsigned off = block_excl_scan<VGF_THREADS>(f[0] + f[1], s_warp, tile_total);
            unsigned slot = slot_base + off;
#pragma unroll
            for (int j = 0; j < VGF_IPT; ++j) {
                if (!f[j]) continue;
                // centroid of the voxel that starts at item i0 + j: sequential fp32 sums over the contiguous sorted points (ascending input
                // index within a voxel: the sort is stable), divided by (float)count; the segment ends where the key changes
                const unsigned b = (unsigned)(i0 + j);
                const unsigned key = __ldcg(kin + b);
                float sx = 0.f, sy = 0.f, sz = 0.f, si = 0.f;
                unsigned k = b; bool open = true;
                while (open) {
                    float4 p[8]; unsigned kk[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) { const unsigned idx = k + u; const bool in = idx < (unsigned)n; kk[u] = in ? __ldcg(kin + idx) : ~key; p[u] = in ? __ldcg(a.pts_sorted + idx) : make_float4(0.f, 0.f, 0.f, 0.f); }
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        if (open && kk[u] == key) { sx += p[u].x; sy += p[u].y; sz += p[u].z; si += p[u].w; ++k; }
                        else open = false;
                    }
                }
                const float cn = (float)(k - b);
                a.seg_start[slot] = b;
                a.out[slot] = make_float4(sx / cn, sy / cn, sz / cn, si / cn);
                if (a.out_keys) a.out_keys[slot] = (int)key;
                if (a.membership) for (unsigned m2 = b; m2 < k; ++m2) a.membership[__ldcg(vin + m2)] = (int)slot;
                ++slot;
            }
            slot_base += tile_total;
        }
    }
    stamp();
    vgf_finish(a.bar);
}

// out must hold cnt.bound points.  n_out_dev receives the voxel count (device int).
// coop_grid > 0: clouds beyond the single-CTA size take the one-kernel cooperative path on that many CTAs (one per SM).
inline int voxel_grid_device(const float4* in, Count cnt, float leaf, float4* out, int* n_out_dev, int* membership, int* out_keys,
                             VoxelGridWork& w, cudaStream_t s, int coop_grid = 0) {
    const int nb = cnt.bound;
    if (nb <= 0) { CUDA_TRY(cudaMemsetAsync(n_out_dev, 0, sizeof(int), s)); w.last_launches = 1; return LIORF_OK; }
    int rc;
    w.last_launches = 10;                                           // multi-kernel path: memset + minmax + keys + hist + 4 passes + head scan + centroids
    // (clouds of more than four tiles per CTA keep the multi-kernel path: a chunk of several tiles is swept twice per pass, and the
    // one-kernel version was measured slower there — 0.47 against 0.29 ms for 2.3 M points on 132 CTAs, 0.23 against 0.15 ms for 650 k on
    // 64 — while at two tiles per CTA it is still ahead: the look-ahead front end's 24 k-point bound on 16 CTAs, 0.040 against 0.069 ms)
    if (coop_grid > 0 && w.fused_bar && !w.force_multi && ((nb > VGS_CAP && nb <= 4 * coop_grid * VGF_TILE) || w.force_large)) {
        if ((rc = w.keys.reserve(nb)) || (rc = w.sort.keys_alt.reserve(nb)) || (rc = w.sort.vals_a.reserve(nb)) || (rc = w.sort.vals_b.reserve(nb)) ||
            (rc = w.seg_start.reserve((size_t)nb + 1)) || (rc = w.pts_sorted.reserve(nb)) || (rc = w.partial.reserve((size_t)coop_grid * 6)) ||
            (rc = w.cta_hist.reserve((size_t)coop_grid * RADIX)) || (rc = w.cta_heads.reserve(coop_grid))) return rc;
        VgFusedArgs a;
        a.pts = in; a.cnt = cnt; a.leaf = leaf; a.out = out; a.n_out = n_out_dev; a.membership = membership; a.out_keys = out_keys; a.meta = w.meta;
        a.keys_a = w.keys.p; a.keys_b = w.sort.keys_alt.p; a.vals_a = w.sort.vals_a.p; a.vals_b = w.sort.vals_b.p;
        a.pts_sorted = w.pts_sorted.p; a.seg_start = w.seg_start.p; a.partial_mm = w.partial.p; a.cta_hist = w.cta_hist.p; a.cta_heads = w.cta_heads.p;
        a.bar = w.fused_bar; a.err_flag = w.err_flag; a.dbg = w.dbg;
        void* args[] = {&a};
        static const bool plain_launch = std::getenv("LIORF_VG_PLAIN_LAUNCH") != nullptr;     // experiment: launch latency of a cooperative launch
        if (plain_launch) k_vg_fused<<<coop_grid, VGF_THREADS, 0, s>>>(a);
        else CUDA_TRY(cudaLaunchCooperativeKernel((void*)k_vg_fused, dim3(coop_grid), dim3(VGF_THREADS), args, 0, s));
        w.last_launches = 1;
        return LIORF_OK;
    }
    if (nb <= VGS_CAP && !w.force_large) {
        if ((rc = w.seg_start.reserve((size_t)nb + 1))) return rc;
        if (!w.small_attr_set) { CUDA_TRY(cudaFuncSetAttribute(k_vg_small, cudaFuncAttributeMaxDynamicSharedMemorySize, VGS_SMEM)); w.small_attr_set = true; }
        k_vg_small<<<1, VGS_THREADS, VGS_SMEM, s>>>(in, cnt, leaf, out, n_out_dev, membership, out_keys, w.meta, w.seg_start.p);
        w.last_launches = 1;
        CUDA_TRY(cudaGetLastError());
        return LIORF_OK;
    }
    int mmb = (nb + VG_MM_BLOCK * 8 - 1) / (VG_MM_BLOCK * 8); if (mmb > kNumSMs) mmb = kNumSMs;
    if ((rc = w.partial.reserve((size_t)mmb * 6))) return rc;
    if ((rc = w.keys.reserve(nb))) return rc;
    if ((rc = w.seg_start.reserve((size_t)nb + 1))) return rc;
    k_vg_minmax<<<mmb, VG_MM_BLOCK, 0, s>>>(in, cnt, leaf, w.partial.p, w.mm_counter, w.meta);
    k_vg_keys<<<(nb + 255) / 256, 256, 0, s>>>(in, cnt, w.meta, w.keys.p);
    unsigned* sorted_idx = nullptr;
    if ((rc = radix_sort_pairs_iota(w.keys.p, cnt, w.sort, &sorted_idx, s))) return rc;
    if ((rc = launch_scan(cnt, VgHeadLoad{w.keys.p}, VgHeadStore{w.seg_start.p, cnt}, w.scan, (unsigned*)n_out_dev, s))) return rc;
    k_vg_centroid<<<(nb + 127) / 128, 128, 0, s>>>(in, sorted_idx, w.seg_start.p, (const unsigned*)n_out_dev, out, membership, w.keys.p, out_keys);
    CUDA_TRY(cudaGetLastError());
    return LIORF_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Segmented VoxelGrid: S independent clouds ("segments", contiguous in one array) filtered in one pass, each exactly as
// voxel_grid_device filters it alone — PCL's per-cloud min_b / div_b, the int32 overflow guard per segment (a segment that trips it
// passes through unchanged), centroids summed sequentially in input order within each (segment, voxel).
//   k_vgseg_bounds : per-segment min/max over host-planned tiles that never straddle two segments (order-independent atomics)
//   k_vgseg_meta   : one thread per segment derives its VoxMeta and key range (div_b product, or the point count under the guard);
//                    seg_base = exclusive prefix of the ranges, flags a total beyond 2^32
//   k_vgseg_keys   : key = seg_base[segment] + PCL voxel index, so one 32-bit stable sort orders by (segment, voxel)
//   then the multi-kernel path's radix sort, head scan and k_vg_centroid unchanged, and
//   k_vgseg_out    : each segment's first voxel and voxel count (binary search of seg_base in the sorted voxel keys)
// ---------------------------------------------------------------------------------------------------------------
constexpr int VGSEG_TILE = 4096;
struct VgSegTile { int seg, begin, end, pad; };

__device__ __forceinline__ unsigned vgseg_ord(float f) {           // order-preserving float → unsigned (min/max by integer atomics)
    const unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float vgseg_unord(unsigned u) { return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u); }

// mn[3 s + a] = encoded min (initialised to 0xffffffff), mx[3 s + a] = encoded max (initialised to 0)
__global__ void __launch_bounds__(256) k_vgseg_bounds(const float4* __restrict__ pts, const VgSegTile* __restrict__ tiles, unsigned* __restrict__ mn_enc,
                                                      unsigned* __restrict__ mx_enc) {
    const VgSegTile t = tiles[blockIdx.x];
    float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int i = t.begin + (int)threadIdx.x; i < t.end; i += blockDim.x) {
        const float4 p = pts[i];
        mn[0] = fminf(mn[0], p.x); mx[0] = fmaxf(mx[0], p.x);
        mn[1] = fminf(mn[1], p.y); mx[1] = fmaxf(mx[1], p.y);
        mn[2] = fminf(mn[2], p.z); mx[2] = fmaxf(mx[2], p.z);
    }
    __shared__ float s_red[8][6];
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { mn[a] = fminf(mn[a], __shfl_xor_sync(FULL, mn[a], o)); mx[a] = fmaxf(mx[a], __shfl_xor_sync(FULL, mx[a], o)); }
    if (lane_id() == 0) { for (int a = 0; a < 3; ++a) { s_red[warp_id()][a] = mn[a]; s_red[warp_id()][3 + a] = mx[a]; } }
    __syncthreads();
    if (threadIdx.x < 6) {
        float v = s_red[0][threadIdx.x];
        for (int w = 1; w < (int)blockDim.x / 32; ++w) v = threadIdx.x < 3 ? fminf(v, s_red[w][threadIdx.x]) : fmaxf(v, s_red[w][threadIdx.x]);
        if (threadIdx.x < 3) atomicMin(mn_enc + t.seg * 3 + threadIdx.x, vgseg_ord(v)); else atomicMax(mx_enc + t.seg * 3 + threadIdx.x - 3, vgseg_ord(v));
    }
}

// one block; S <= any size (threads stride), then thread 0 forms the prefix of the ranges
__global__ void __launch_bounds__(1024) k_vgseg_meta(const int* __restrict__ seg_n, int S, const unsigned* __restrict__ mn_enc, const unsigned* __restrict__ mx_enc, float leaf, VoxMeta* __restrict__ metas,
                                                     unsigned long long* __restrict__ seg_base, int* __restrict__ range_overflow) {
    for (int s = threadIdx.x; s < S; s += blockDim.x) {
        const int n = seg_n[s];
        float mn[3], mx[3];
        for (int a = 0; a < 3; ++a) { mn[a] = n > 0 ? vgseg_unord(mn_enc[s * 3 + a]) : 0.f; mx[a] = n > 0 ? vgseg_unord(mx_enc[s * 3 + a]) : 0.f; }
        VoxMeta m;                                                    // k_vg_minmax's arithmetic
        m.n = n;
        m.inv = 1.0f / leaf;
        long long d[3];
        for (int a = 0; a < 3; ++a) {
            m.minp[a] = mn[a]; m.maxp[a] = mx[a];
            d[a] = (long long)((mx[a] - mn[a]) * m.inv) + 1;
            m.min_b[a] = (int)floorf(mn[a] * m.inv);
            const int max_b = (int)floorf(mx[a] * m.inv);
            m.div_b[a] = max_b - m.min_b[a] + 1;
        }
        m.overflow = (n > 0 && d[0] * d[1] * d[2] > 2147483647LL) ? 1 : 0;
        m.mul1 = m.div_b[0]; m.mul2 = m.div_b[0] * m.div_b[1];
        metas[s] = m;
        seg_base[s] = n <= 0 ? 0ull : m.overflow ? (unsigned long long)n : (unsigned long long)((long long)m.div_b[0] * m.div_b[1] * m.div_b[2]);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long run = 0;
        for (int s = 0; s < S; ++s) { const unsigned long long r = seg_base[s]; seg_base[s] = run; run += r; }
        seg_base[S] = run;
        *range_overflow = run > (1ull << 32) ? 1 : 0;
    }
}

__global__ void __launch_bounds__(256) k_vgseg_keys(const float4* __restrict__ pts, const VgSegTile* __restrict__ tiles, const int* __restrict__ seg_first,
                                                    const VoxMeta* __restrict__ metas, const unsigned long long* __restrict__ seg_base, unsigned* __restrict__ keys) {
    const VgSegTile t = tiles[blockIdx.x];
    const VoxMeta& m = metas[t.seg];
    const unsigned base = (unsigned)seg_base[t.seg];
    const int first = seg_first[t.seg];
    const float inv = m.inv;
    for (int i = t.begin + (int)threadIdx.x; i < t.end; i += blockDim.x) {
        if (m.overflow) { keys[i] = base + (unsigned)(i - first); continue; }      // every point its own voxel ⇒ output == input
        keys[i] = base + vgf_key(pts[i], inv, m.min_b[0], m.min_b[1], m.min_b[2], m.mul1, m.mul2);
    }
}

// seg_vox[2 s] = first voxel of segment s in the output, seg_vox[2 s + 1] = its voxel count
__global__ void __launch_bounds__(256) k_vgseg_out(const unsigned* __restrict__ sorted_keys, const unsigned* __restrict__ seg_start, const unsigned* __restrict__ n_out,
                                                   const unsigned long long* __restrict__ seg_base, int S, int* __restrict__ seg_vox) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const int nv = (int)*n_out;
    auto lower = [&](unsigned long long key) {                    // first voxel whose key >= key
        int lo = 0, hi = nv;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if ((unsigned long long)sorted_keys[seg_start[mid]] < key) lo = mid + 1; else hi = mid; }
        return lo;
    };
    const int b = lower(seg_base[s]), e = lower(seg_base[s + 1]);
    seg_vox[2 * s] = b; seg_vox[2 * s + 1] = e - b;
}

}  // namespace liorf
