// sc_tensor.cuh — ScanContext ring-key search (detectLoopClosureID stage 1, include/Scancontext.cpp:289-295) as a dense
// contraction on the 5th-generation tensor cores (tcgen05.mma, accumulators in TMEM, operands staged by TMA bulk copies).
//
// The reference asks a kd-tree for the exact 3 nearest 20-D fp32 ring keys (nanoflann, include/nanoflann.hpp:383-408).
// A GEMM cannot reproduce nanoflann's fp32 operation order, so the tensor cores are used as a PROVABLY COMPLETE coarse
// filter and the survivors are re-ranked with the exact arithmetic:
//
//   d~(q,k) = |x|^2 + |y|^2 - 2 x.y ,  x = q - c, y = k - c (c = database mean: shrinks the norms, hence the error)
//   every fp32 value is split in two bf16 terms (hi + lo); the three significant cross terms, the two norms (split
//   likewise) and the constant 1s are laid along ONE contraction axis of length 64:
//       A row (query):  [ xh(20) | xh(20) | xl(20) | nxh nxl 1 1 ]
//       B row (key)  :  [-2yh(20)|-2yl(20)|-2yh(20)| 1 1 nyh nyl ]
//   so one 128x128x64 bf16 MMA chain with fp32 accumulation in TMEM yields d~ directly.
//   |d~ - d| <= eps(q,k) = 2^-13 (|x|^2 + |y|^2)   (split truncation 3*2^-18, norm split 2^-17, accumulation budget
//   2^-14; tests/test_gpu_sc_tensor.py measures the real error over millions of pairs and asserts a 4x margin).
//
//   k_sc_tensor : the GEMM; its epilogue reduces every 32 consecutive accumulator columns (a "chunk" = 32 keys) to their
//                 minimum and stores only the minima: per chunk (cmin32) and per 128-key tile (cmin, what the selection streams)
//   k_sct_top3 / k_sct_select: per query t3 = 3rd smallest chunk minimum (three different chunks hold three different keys,
//                 so t3 bounds the 3rd smallest d~ from above), then every chunk with cmin32 <= t3 + 2 eps_max(q) is a candidate
//   k_sct_rerank: exact nanoflann-order distances of the <= 32 keys of each candidate chunk, top-3 by (dist, idx)
//   Completeness: the exact 3rd-best distance d3 <= t3 + eps (three different keys have d~ <= t3, hence exact distance
//   <= t3 + eps), and a key of the exact top-3 has d~ <= d + eps <= d3 + eps <= t3 + 2 eps  =>  its chunk is a candidate.
//   A query with more than SCT_CAP candidate chunks is answered by an exact scan of all keys instead (same warp of
//   k_sct_rerank) — never a wrong answer.
//
// Kernel shape (k_sc_tensor): persistent, one CTA per SM, 320 threads:
//   warp 0     TMA producer: 16 KB operand images with cp.async.bulk + mbarrier complete_tx (6-stage key ring, 2 query buffers)
//   warp 1     one lane issues tcgen05.mma (M=128,N=128,K=16 x4 k-steps x2 query sub-tiles per step), tcgen05.commit
//   warps 2-9  epilogue (one 128x128 accumulator each): 4 x tcgen05.ld 32x32b.x32 in flight, min trees, 4 coalesced stores
//   TMEM: 2 accumulator stages x (2 sub-tiles x 128 columns) = 512 columns.
// The work list is the linearised (256-query tile, 128-key tile) grid cut into gridDim equal runs; a CTA keeps the two
// query images resident and streams key images, so each key image is read from L2 once per 256 queries.
#pragma once
#include <cuda_bf16.h>
#include <cstdint>
#include "scancontext.cuh"
#include "sc_window.cuh"

namespace liorf {

constexpr int SCT_SUB = 128;                       // MMA M (queries per sub-tile) and N (keys per step)
constexpr int SCT_QT = 2 * SCT_SUB;                // queries per CTA segment
constexpr int SCT_KT = 128;                        // keys per step
constexpr int SCT_KDIM = 64;                       // contraction length
constexpr int SCT_TILE_BYTES = SCT_SUB * SCT_KDIM * 2;     // 16 KB operand image (128 rows x 64 bf16)
constexpr int SCT_STAGES = 6;
constexpr int SCT_CAP = 64;                        // candidate chunks (of 32 keys) kept per query
constexpr int SCT_CHUNK = 32;                      // accumulator columns (keys) per candidate chunk; 4 chunks per key tile
constexpr int SCT_THREADS = 320;                   // producer warp, MMA warp, 8 epilogue warps
constexpr float SCT_EPS_REL = 1.0f / 8192.0f;      // eps(q,k) = 2^-13 (|x|^2 + |y|^2)
// operand image = the canonical K-major SWIZZLE_128B shared-memory layout (what TMA writes for a 64-element bf16 box):
// one 128-byte row per query/key, 8-row groups of 1024 B, 16-byte chunk c of row r stored at chunk position c ^ (r % 8)
constexpr uint32_t SCT_SBO = 1024;
constexpr int SCT_SMEM = 1024 + 4 * SCT_TILE_BYTES + SCT_STAGES * SCT_TILE_BYTES + 256;

// ---------------------------------------------------------------------------------------------------------------
// operand images
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned short bf16_bits(float f) { return __bfloat16_as_ushort(__float2bfloat16_rn(f)); }
__device__ __forceinline__ float bf16_val(unsigned short b) { return __uint_as_float((unsigned)b << 16); }

__global__ void __launch_bounds__(1024) k_sct_center(const float* __restrict__ keys, int n, float* __restrict__ center) {
    __shared__ double s_part[32][SC_RING];
    double acc[SC_RING];
#pragma unroll
    for (int d = 0; d < SC_RING; ++d) acc[d] = 0.0;
    for (int r = threadIdx.x; r < n; r += blockDim.x) {
        const float4* p = reinterpret_cast<const float4*>(keys + (size_t)SC_RING * r);
#pragma unroll
        for (int g = 0; g < 5; ++g) { float4 v = __ldg(p + g); acc[4 * g] += v.x; acc[4 * g + 1] += v.y; acc[4 * g + 2] += v.z; acc[4 * g + 3] += v.w; }
    }
#pragma unroll
    for (int d = 0; d < SC_RING; ++d) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[d] += __shfl_xor_sync(FULL, acc[d], o);
    }
    if (lane_id() == 0) for (int d = 0; d < SC_RING; ++d) s_part[warp_id()][d] = acc[d];
    __syncthreads();
    if (threadIdx.x < SC_RING) {
        double s = 0; for (int w = 0; w < (int)(blockDim.x / 32); ++w) s += s_part[w][threadIdx.x];
        center[threadIdx.x] = n > 0 ? (float)(s / n) : 0.f;
    }
}

// one thread per image row.  IS_KEY: B image, rows = keys padded to nkt * 128 with never-selected rows; image position
// p = tile * 128 + col holds key (col * nkt + tile), so keys adjacent in the database (similar ring keys along a drive)
// land in different tiles and the per-32-column minima the epilogue tracks stay decorrelated.  Otherwise A image,
// rows = queries in order, padded to a multiple of 256 with zero rows.
template <bool IS_KEY>
__global__ void __launch_bounds__(128) k_sct_image(const float* __restrict__ vecs, int n, int n_pad, int nkt, const float* __restrict__ center,
                                                  uint8_t* __restrict__ img, float* __restrict__ norm_out, unsigned* __restrict__ nmax_bits) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pad) return;
    const int r = IS_KEY ? (p % SCT_SUB) * nkt + p / SCT_SUB : p;
    unsigned short v[SCT_KDIM];
#pragma unroll
    for (int k = 0; k < SCT_KDIM; ++k) v[k] = 0;
    const unsigned short ONE = 0x3f80;
    if (r < n) {
        double acc = 0.0;
#pragma unroll
        for (int d = 0; d < SC_RING; ++d) {
            const float x = __ldg(vecs + (size_t)SC_RING * r + d) - __ldg(center + d);
            acc += (double)x * (double)x;
            const unsigned short h = bf16_bits(x);
            const unsigned short l = bf16_bits(x - bf16_val(h));
            if (IS_KEY) {
                const unsigned short h2 = bf16_bits(-2.f * bf16_val(h)), l2 = bf16_bits(-2.f * bf16_val(l));
                v[d] = h2; v[20 + d] = l2; v[40 + d] = h2;
            } else { v[d] = h; v[20 + d] = h; v[40 + d] = l; }
        }
        const float nrm = (float)acc;
        const unsigned short nh = bf16_bits(nrm), nl = bf16_bits(nrm - bf16_val(nh));
        if (IS_KEY) { v[60] = ONE; v[61] = ONE; v[62] = nh; v[63] = nl; }
        else { v[60] = nh; v[61] = nl; v[62] = ONE; v[63] = ONE; }
        if (norm_out) norm_out[r] = nrm;
        if (nmax_bits) atomicMax(nmax_bits, __float_as_uint(nrm));
    } else if (IS_KEY) v[62] = bf16_bits(1e30f);
    const int row = p % SCT_SUB;
    uint8_t* base = img + (size_t)(p / SCT_SUB) * SCT_TILE_BYTES + (size_t)row * 128;
#pragma unroll
    for (int kc = 0; kc < 8; ++kc) {
        uint4 w;
        w.x = v[8 * kc] | ((unsigned)v[8 * kc + 1] << 16); w.y = v[8 * kc + 2] | ((unsigned)v[8 * kc + 3] << 16);
        w.z = v[8 * kc + 4] | ((unsigned)v[8 * kc + 5] << 16); w.w = v[8 * kc + 6] | ((unsigned)v[8 * kc + 7] << 16);
        *reinterpret_cast<uint4*>(base + ((kc ^ (row & 7)) << 4)) = w;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// PTX wrappers (sm_100a)
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// bounded wait: a protocol bug must end the kernel with an error flag, never hang the device
__device__ __forceinline__ bool mbar_wait(uint32_t bar, uint32_t parity, volatile int* s_abort, int* err_flag) {
    for (uint32_t it = 0; it < (1u << 21); ++it) {
        if (mbar_try_wait(bar, parity)) return true;
        if ((it & 255u) == 255u && *s_abort) return false;
    }
    *s_abort = 1; atomicCAS(err_flag, 0, 5);                      // 5: an mbarrier (TMA copy / tensor-core commit) never completed
    return false;
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) { asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b),
                 "r"(idesc), "r"(accumulate) : "memory");
}
// shared-memory matrix descriptor, K-major SWIZZLE_128B: start>>4 [0,14), LBO>>4 [16,30) (unused for swizzled K-major: 1),
// SBO>>4 [32,46) = 1024 B between 8-row groups, version 1 [46,48), layout type 2 [61,64).  A k-step of 16 bf16 advances the
// start address by 32 B inside the swizzle atom.
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr) {
    return (uint64_t)((addr & 0x3ffffu) >> 4) | (1ull << 16) | ((uint64_t)(SCT_SBO >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// instruction descriptor: D fp32 [4,6)=1, A bf16 [7,10)=1, B bf16 [10,13)=1, both K-major, N>>3 [17,23), M>>4 [24,29)
constexpr uint32_t SCT_IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(SCT_KT >> 3) << 17) | ((uint32_t)(SCT_SUB >> 4) << 24);

// One step's tensor-core work issued by ONE elected lane from warp-uniform operands: 2 query sub-tiles x 4 k-steps of
// M128 N128 K16, then the commits.  Everything the issue needs is computed by the whole warp in uniform code, so the
// descriptors stay in uniform registers (a single lane re-deriving them costs ~150 cycles per MMA in register moves and
// makes the issue loop, not the tensor core, the bottleneck).
__device__ __forceinline__ void tc_issue_step(uint32_t td, uint64_t da, uint64_t db, uint32_t bar_b_empty, uint32_t bar_t_full, uint32_t bar_a_empty, uint32_t seg_end) {
    asm volatile(
        "{\n\t"
        ".reg .pred pe, pz, po, pa;\n\t"
        ".reg .b64 a1, a2, a3, a4, a5, a6, a7, b1, b2, b3;\n\t"
        ".reg .b32 t1;\n\t"
        "elect.sync _|pe, 0xffffffff;\n\t"
        "setp.ne.b32 pz, 0, 0;\n\t"
        "setp.eq.b32 po, 0, 0;\n\t"
        "setp.ne.and.b32 pa, %5, 0, pe;\n\t"
        "add.u64 a1, %1, 2;\n\t add.u64 a2, %1, 4;\n\t add.u64 a3, %1, 6;\n\t"
        "add.u64 a4, %1, 1024;\n\t add.u64 a5, %1, 1026;\n\t add.u64 a6, %1, 1028;\n\t add.u64 a7, %1, 1030;\n\t"
        "add.u64 b1, %2, 2;\n\t add.u64 b2, %2, 4;\n\t add.u64 b3, %2, 6;\n\t"
        "add.u32 t1, %0, 128;\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, pz;\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [t1], a4, %2, %3, pz;\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], a1, b1, %3, po;\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [t1], a5, b1, %3, po;\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], a2, b2, %3, po;\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [t1], a6, b2, %3, po;\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], a3, b3, %3, po;\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [t1], a7, b3, %3, po;\n\t"
        "@pe tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%4];\n\t"
        "@pe tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%6];\n\t"
        "@pa tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%7];\n\t"
        "}\n"
        ::"r"(td), "l"(da), "l"(db), "r"(SCT_IDESC), "r"(bar_b_empty), "r"(seg_end), "r"(bar_t_full), "r"(bar_a_empty) : "memory");
}

#define SCT_R32(v) "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), \
    "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), \
    "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
#define SCT_RW32(v) "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), \
    "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]), "+r"(v[16]), "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]), \
    "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
// 32 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, "
                 "%24, %25, %26, %27, %28, %29, %30, %31}, [%32];" : SCT_R32(v) : "r"(taddr) : "memory");
}
// the registers of an earlier tmem_ld32 become valid here; tying them to the wait keeps every use after it
__device__ __forceinline__ void tmem_wait_ld(uint32_t (&v)[32]) { asm volatile("tcgen05.wait::ld.sync.aligned;" : SCT_RW32(v) : : "memory"); }

__device__ __forceinline__ void tmem_wait_ld4(uint32_t (&a)[32], uint32_t (&b)[32], uint32_t (&c)[32], uint32_t (&d)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;" : SCT_RW32(a) : : "memory");
    asm volatile("" : SCT_RW32(b) : : "memory");
    asm volatile("" : SCT_RW32(c) : : "memory");
    asm volatile("" : SCT_RW32(d) : : "memory");
}
// 2-input minimum tree (FMNMX on the ALU pipe; the 3-input FMNMX3 form issues at a fraction of that rate)
__device__ __forceinline__ float min32(const uint32_t (&v)[32]) {
    float m[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) m[i] = fminf(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1]));
#pragma unroll
    for (int w = 8; w > 0; w >>= 1) {
#pragma unroll
        for (int i = 0; i < w; ++i) m[i] = fminf(m[i], m[i + w]);
    }
    return m[0];
}
__device__ __forceinline__ void top3_min_update(float m, float& t1, float& t2, float& t3) {
    const float b = fmaxf(m, t1); t1 = fminf(m, t1);
    const float e = fmaxf(b, t2); t2 = fminf(b, t2);
    t3 = fminf(e, t3);
}

struct SctArgs {
    const uint8_t* a_img;      // [n_sqt][2][SCT_TILE_BYTES]
    const uint8_t* b_img;      // [nkt][SCT_TILE_BYTES]
    int Q, n_keys, nkt, n_sqt;
    float* cmin;               // out: [nkt][n_sqt * SCT_QT]      minimum d~ over the 128 keys of each tile (streamed by the selection)
    float* cmin32;             // out: [nkt * 4][n_sqt * SCT_QT]  minimum d~ of each 32-key chunk (read only for tiles that pass)
    float* dump;               // DUMP (tests): every d~, [n_sqt * SCT_QT][nkt * SCT_KT] indexed by database key
    int* err_flag;
    const int* lim;            // LIM: [Q] query q sees only keys [0, lim[q])
};

__device__ __forceinline__ long long sct_first_step(int cta, long long total, int grid) { return (long long)cta * total / grid; }

// LIM (batched detectLoopClosureID, a.lim): query q sees only keys [0, lim[q]).  Key tiles interleave the keys (column i of tile kt is key
// i * nkt + kt), so that prefix is a column prefix in every tile: q keeps the first ceil((lim[q] - kt) / nkt) columns of tile kt.  The epilogue
// sets the other columns to +inf before its min trees — never to 3.0e38f, which the selection's `<= thr` could pass — so the masked minima
// feed k_sct_top3 / k_sct_select unchanged: three chunks with finite masked minima still hold three distinct keys of the prefix.
template <bool DUMP, bool LIM = false>
__global__ void __launch_bounds__(SCT_THREADS, 1) k_sc_tensor(SctArgs a) {
    extern __shared__ uint8_t sct_smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)sct_smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* sA = smem;                                            // [2 buffers][2 sub-tiles][16 KB]
    uint8_t* sB = smem + 4 * SCT_TILE_BYTES;                       // [SCT_STAGES][16 KB]
    uint64_t* bars = reinterpret_cast<uint64_t*>(sB + SCT_STAGES * SCT_TILE_BYTES);
    constexpr int A_FULL = 0, A_EMPTY = 2, B_FULL = 4, B_EMPTY = B_FULL + SCT_STAGES, T_FULL = B_EMPTY + SCT_STAGES, T_EMPTY = T_FULL + 2, NBAR = T_EMPTY + 2;
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bars + NBAR);
    volatile int* s_abort = reinterpret_cast<volatile int*>(s_tmem + 1);
    const uint32_t bar0 = smem_u32(bars);
    auto BAR = [&](int i) { return bar0 + 8u * (uint32_t)i; };

    const int warp = warp_id(), lane = lane_id();
    const long long total = (long long)a.n_sqt * a.nkt;
    const long long s_begin = sct_first_step(blockIdx.x, total, gridDim.x), s_end = sct_first_step(blockIdx.x + 1, total, gridDim.x);
    const int sqt0 = (int)(s_begin / a.nkt), kt0 = (int)(s_begin % a.nkt);          // the only division: the roles step (sqt, kt) incrementally

    if (threadIdx.x == 0) {
        *s_abort = 0;
        for (int i = 0; i < 2; ++i) { mbar_init(BAR(A_FULL + i), 1); mbar_init(BAR(A_EMPTY + i), 1); mbar_init(BAR(T_FULL + i), 1); mbar_init(BAR(T_EMPTY + i), 8); }
        for (int i = 0; i < SCT_STAGES; ++i) { mbar_init(BAR(B_FULL + i), 1); mbar_init(BAR(B_EMPTY + i), 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;
    const int n_steps = (int)(s_end - s_begin);

    // The producer and MMA loops run on ALL lanes of their warp (uniform control flow keeps counters, addresses and
    // descriptors in uniform registers); only the asynchronous issue itself is done by one elected lane.
    if (warp == 0) {
        // ===== TMA producer =====
        int seg = 0, sqt = sqt0, kt = kt0, st = 0; uint32_t ph = 1;                 // ph: parity to wait for on B_EMPTY[st] (first lap passes)
        for (int it = 0; it < n_steps; ++it) {
            if (it == 0 || kt == 0) {
                const int ab = seg & 1;
                if (!mbar_wait(BAR(A_EMPTY + ab), ((seg >> 1) & 1) ^ 1, s_abort, a.err_flag)) break;
                if (lane == 0) {
                    mbar_expect_tx(BAR(A_FULL + ab), 2 * SCT_TILE_BYTES);
                    bulk_g2s(smem_u32(sA) + ab * 2 * SCT_TILE_BYTES, a.a_img + (size_t)sqt * 2 * SCT_TILE_BYTES, 2 * SCT_TILE_BYTES, BAR(A_FULL + ab));
                }
                ++seg;
            }
            if (!mbar_wait(BAR(B_EMPTY + st), ph, s_abort, a.err_flag)) break;
            if (lane == 0) {
                mbar_expect_tx(BAR(B_FULL + st), SCT_TILE_BYTES);
                bulk_g2s(smem_u32(sB) + st * SCT_TILE_BYTES, a.b_img + (size_t)kt * SCT_TILE_BYTES, SCT_TILE_BYTES, BAR(B_FULL + st));
            }
            if (++st == SCT_STAGES) { st = 0; ph ^= 1; }
            if (++kt == a.nkt) { kt = 0; ++sqt; }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        int seg = -1, kt = kt0, st = 0; uint32_t ph = 0;                            // ph: parity to wait for on B_FULL[st]
        const uint64_t da0 = smem_desc(smem_u32(sA)), db0 = smem_desc(smem_u32(sB));   // descriptors advance by (bytes >> 4) in the low word
        for (int it = 0; it < n_steps; ++it) {
            if (it == 0 || kt == 0) {
                ++seg;
                if (!mbar_wait(BAR(A_FULL + (seg & 1)), (seg >> 1) & 1, s_abort, a.err_flag)) break;
            }
            const int ab = seg & 1, acc = it & 1;
            if (!mbar_wait(BAR(B_FULL + st), ph, s_abort, a.err_flag)) break;
            if (!mbar_wait(BAR(T_EMPTY + acc), ((it >> 1) & 1) ^ 1, s_abort, a.err_flag)) break;
            tc_fence_after();
            const bool seg_end = (it + 1 == n_steps) || (kt == a.nkt - 1);
            tc_issue_step(tmem_base + acc * 256, da0 + (uint64_t)(ab * (2 * SCT_TILE_BYTES >> 4)), db0 + (uint64_t)(st * (SCT_TILE_BYTES >> 4)),
                          BAR(B_EMPTY + st), BAR(T_FULL + acc), BAR(A_EMPTY + ab), seg_end ? 1u : 0u);
            __syncwarp();
            if (++st == SCT_STAGES) { st = 0; ph ^= 1; }
            if (++kt == a.nkt) kt = 0;
        }
    } else {
        // ===== epilogue: 8 warps; TMEM lane quadrant = warp % 4, query sub-tile j = (warp - 2) / 4 =====
        // Two warps share each SM sub-partition, so one warp's TMEM loads overlap the other's min tree.
        const int qd = warp & 3, j = (warp - 2) >> 2;
        const int row = 32 * qd + lane;
        const uint32_t t_lane = tmem_base + ((uint32_t)(32 * qd) << 16) + j * SCT_SUB;
        const size_t n_rows = (size_t)a.n_sqt * SCT_QT;
        int sqt = sqt0, kt = kt0;
        int lim_a = 0, lim_b = 0;                                  // LIM: this row's limit = lim_a * nkt + lim_b → tile kt keeps lim_a + (kt < lim_b) columns
        for (int it = 0; it < n_steps; ++it) {
            const int q = sqt * SCT_QT + j * SCT_SUB + row;
            const int acc = it & 1;
            if (LIM && (it == 0 || kt == 0)) { const int L = q < a.Q ? __ldg(a.lim + q) : 0; lim_a = L / a.nkt; lim_b = L % a.nkt; }
            if (!mbar_wait(BAR(T_FULL + acc), (it >> 1) & 1, s_abort, a.err_flag)) break;
            tc_fence_after();
            const uint32_t tcol = t_lane + acc * 256;
            uint32_t v0[32], v1[32], v2[32], v3[32];
            __syncwarp();
            tmem_ld32(tcol, v0); tmem_ld32(tcol + 32, v1); tmem_ld32(tcol + 64, v2); tmem_ld32(tcol + 96, v3);      // 16 KB per warp in flight
            tmem_wait_ld4(v0, v1, v2, v3);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(BAR(T_EMPTY + acc));        // the values are in registers: release the accumulator stage early
            if constexpr (LIM) {
                const int ncol = lim_a + (kt < lim_b ? 1 : 0);
                if (ncol < SCT_KT) {
                    const uint32_t INF = 0x7f800000u;
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        if (i >= ncol) v0[i] = INF;
                        if (32 + i >= ncol) v1[i] = INF;
                        if (64 + i >= ncol) v2[i] = INF;
                        if (96 + i >= ncol) v3[i] = INF;
                    }
                }
            }
            if (DUMP) {
                float* o = a.dump + (size_t)q * ((size_t)a.nkt * SCT_KT);
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    o[(size_t)i * a.nkt + kt] = __uint_as_float(v0[i]); o[(size_t)(32 + i) * a.nkt + kt] = __uint_as_float(v1[i]);
                    o[(size_t)(64 + i) * a.nkt + kt] = __uint_as_float(v2[i]); o[(size_t)(96 + i) * a.nkt + kt] = __uint_as_float(v3[i]);
                }
            } else {
                const float m0 = min32(v0), m1 = min32(v1), m2 = min32(v2), m3 = min32(v3);
                float* o = a.cmin32 + (size_t)kt * 4 * n_rows + q;             // lanes = consecutive queries: every store is one 128-byte line
                o[0] = m0; o[n_rows] = m1; o[2 * n_rows] = m2; o[3 * n_rows] = m3;
                a.cmin[(size_t)kt * n_rows + q] = fminf(fminf(m0, m1), fminf(m2, m3));
            }
            if (++kt == a.nkt) { kt = 0; ++sqt; }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// Candidate selection on the chunk minima, two small kernels over a (32-query block) x (chunk split) grid so that enough
// 128-byte rows are in flight to stream the minima from L2:
//   k_sct_top3  : partial top-3 of the chunk minima per (query, split)                        → part[split][row][3]
//   k_sct_select: t3(q) = 3rd smallest over the splits (three different chunks hold three different keys, so t3 bounds the
//                 3rd smallest d~ from above); every chunk of this split with cmin <= t3 + 2 eps_max(q),
//                 2 eps_max = 2^-12 (|x|^2 + max_k |y|^2), is appended to the query's candidate list.
constexpr int SCS_SLICES = 8;              // warps per block: each takes every 8th chunk of the block's split
constexpr int SCS_SPLITS = 8;              // chunk ranges (grid.y)
__device__ __forceinline__ void scs_range(int n_chunks, int& c0, int& c1) {
    const int per = (n_chunks + SCS_SPLITS - 1) / SCS_SPLITS;
    c0 = blockIdx.y * per; c1 = min(n_chunks, c0 + per);
}
__global__ void __launch_bounds__(32 * SCS_SLICES) k_sct_top3(const float* __restrict__ cmin, int n_chunks, int n_rows, float* __restrict__ part, int Q, int* __restrict__ cand_cnt,
                                                             int* __restrict__ over_cnt) {
    __shared__ float s_t[SCS_SLICES][3][32];
    const int lane = threadIdx.x & 31, sl = threadIdx.x >> 5;
    const int q = blockIdx.x * 32 + lane;
    if (blockIdx.y == 0 && sl == 0) {                       // arms the selection that follows: candidate counters of these queries, overflow statistic
        if (q < Q) cand_cnt[q] = 0;
        if (blockIdx.x == 0 && lane == 0) *over_cnt = 0;
    }
    const float* col = cmin + q;
    int c0, c1; scs_range(n_chunks, c0, c1);
    float t1 = 3.0e38f, t2 = 3.0e38f, t3 = 3.0e38f;
    int ch = c0 + sl;
    for (; ch + 3 * SCS_SLICES < c1; ch += 4 * SCS_SLICES) {                       // four independent 128-byte rows in flight per warp
        const float a0 = __ldg(col + (size_t)ch * n_rows), a1 = __ldg(col + (size_t)(ch + SCS_SLICES) * n_rows);
        const float a2 = __ldg(col + (size_t)(ch + 2 * SCS_SLICES) * n_rows), a3 = __ldg(col + (size_t)(ch + 3 * SCS_SLICES) * n_rows);
        top3_min_update(a0, t1, t2, t3); top3_min_update(a1, t1, t2, t3); top3_min_update(a2, t1, t2, t3); top3_min_update(a3, t1, t2, t3);
    }
    for (; ch < c1; ch += SCS_SLICES) top3_min_update(__ldg(col + (size_t)ch * n_rows), t1, t2, t3);
    s_t[sl][0][lane] = t1; s_t[sl][1][lane] = t2; s_t[sl][2][lane] = t3;
    __syncthreads();
    if (sl == 0) {
        t1 = t2 = t3 = 3.0e38f;
#pragma unroll
        for (int w = 0; w < SCS_SLICES; ++w) { top3_min_update(s_t[w][0][lane], t1, t2, t3); top3_min_update(s_t[w][1][lane], t1, t2, t3); top3_min_update(s_t[w][2][lane], t1, t2, t3); }
        float* o = part + ((size_t)blockIdx.y * n_rows + q) * 3;
        o[0] = t1; o[1] = t2; o[2] = t3;
    }
}
__device__ __forceinline__ void sct_emit_tile(const float* __restrict__ cmin32, int n_rows, int q, int kt, float thr, int* __restrict__ cand, int* __restrict__ cand_cnt) {
#pragma unroll
    for (int c = 0; c < 4; ++c)
        if (__ldg(cmin32 + (size_t)(4 * kt + c) * n_rows + q) <= thr) {
            const int slot = atomicAdd(cand_cnt + q, 1);
            if (slot < SCT_CAP) cand[(size_t)q * SCT_CAP + slot] = 4 * kt + c;
        }
}
__global__ void __launch_bounds__(32 * SCS_SLICES) k_sct_select(const float* __restrict__ cmin, const float* __restrict__ cmin32, int n_chunks, int n_rows, const float* __restrict__ part,
                                                               const float* __restrict__ qnorm, int Q, const unsigned* __restrict__ nmax_bits,
                                                               int* __restrict__ cand, int* __restrict__ cand_cnt) {
    const int lane = threadIdx.x & 31, sl = threadIdx.x >> 5;
    const int q = blockIdx.x * 32 + lane;
    if (q >= Q) return;
    float thr;
    {
        float t1 = 3.0e38f, t2 = 3.0e38f, t3 = 3.0e38f;
#pragma unroll
        for (int sp = 0; sp < SCS_SPLITS; ++sp) {
            const float* p = part + ((size_t)sp * n_rows + q) * 3;
            top3_min_update(p[0], t1, t2, t3); top3_min_update(p[1], t1, t2, t3); top3_min_update(p[2], t1, t2, t3);
        }
        thr = t3 < 1.0e38f ? t3 + 2.f * SCT_EPS_REL * (qnorm[q] + __uint_as_float(*nmax_bits)) : 3.0e38f;
    }
    const float* col = cmin + q;
    int c0, c1; scs_range(n_chunks, c0, c1);
    int ch = c0 + sl;
    for (; ch + 3 * SCS_SLICES < c1; ch += 4 * SCS_SLICES) {
        const float a0 = __ldg(col + (size_t)ch * n_rows), a1 = __ldg(col + (size_t)(ch + SCS_SLICES) * n_rows);
        const float a2 = __ldg(col + (size_t)(ch + 2 * SCS_SLICES) * n_rows), a3 = __ldg(col + (size_t)(ch + 3 * SCS_SLICES) * n_rows);
        if (fminf(fminf(a0, a1), fminf(a2, a3)) <= thr) {
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float au = u == 0 ? a0 : u == 1 ? a1 : u == 2 ? a2 : a3;
                if (au <= thr) sct_emit_tile(cmin32, n_rows, q, ch + u * SCS_SLICES, thr, cand, cand_cnt);
            }
        }
    }
    for (; ch < c1; ch += SCS_SLICES)
        if (__ldg(col + (size_t)ch * n_rows) <= thr) sct_emit_tile(cmin32, n_rows, q, ch, thr, cand, cand_cnt);
}

// exact re-rank: one warp per query, one lane per key of a candidate chunk; nanoflann's evalMetric op order
// (ringkey_dist_dev), total order (dist, idx).  chunk id = kt * 4 + c holds keys ((32 c + lane) * nkt + kt).
// A query whose candidate list overflowed (> SCT_CAP chunks passed the filter: only adversarial databases do that) is answered by
// the same warp with an exact scan of ALL keys — never a wrong answer.
// Sharded search (sc_shard.cuh, P.enabled): the queries are this rank's slice [P.q0, P.q0 + Q) of the batch and the result — the
// GLOBAL top-3, the keys being the replicated index — goes straight into the candidate array of every rank's window (phase C);
// the last block raises the flags: compute and transfer in ONE kernel.
// LIM (batched detectLoopClosureID): query q sees only keys [0, lim[q]): candidate keys past it are skipped, the overflow scan stops there.
template <bool LIM>
__global__ void __launch_bounds__(256) k_sct_rerank(const float* __restrict__ keys, int n_keys, int nkt, int idx_offset, const float* __restrict__ qkeys, int Q,
                                                   const int* __restrict__ cand, const int* __restrict__ cand_cnt, float* __restrict__ out_d, int* __restrict__ out_i,
                                                   int* __restrict__ over_cnt, ShardPush P, const int* __restrict__ lim) {
    const int q = blockIdx.x * (blockDim.x / 32) + warp_id();
    const int l = lane_id();
    if (q < Q) {
        if (LIM) n_keys = lim[q];
        const int n = cand_cnt[q];
        float aq[20];
#pragma unroll
        for (int k = 0; k < 20; ++k) aq[k] = __ldg(qkeys + 20 * (size_t)q + k);
        Top3 t; top3_init(t);
        if (n > SCT_CAP) {
            if (l == 0) atomicAdd(over_cnt, 1);
            for (int kidx = l; kidx < n_keys; kidx += 32) top3_insert(t, ringkey_dist_dev(aq, reinterpret_cast<const float4*>(keys + 20 * (size_t)kidx)), idx_offset + kidx);
        } else {
            for (int i = 0; i < n; ++i) {
                const int ch = cand[(size_t)q * SCT_CAP + i];
                const int kidx = (SCT_CHUNK * (ch & 3) + l) * nkt + (ch >> 2);
                if (kidx < n_keys) top3_insert(t, ringkey_dist_dev(aq, reinterpret_cast<const float4*>(keys + 20 * (size_t)kidx)), idx_offset + kidx);
            }
        }
        float rd = INFINITY; int ri = 0x7fffffff;                  // lane r < 3 ends up holding the r-th best
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            float md = t.d[0]; int mi = t.i[0];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float od = __shfl_xor_sync(FULL, md, o); const int oi = __shfl_xor_sync(FULL, mi, o);
                if (od < md || (od == md && oi < mi)) { md = od; mi = oi; }
            }
            if (t.d[0] == md && t.i[0] == mi) { t.d[0] = t.d[1]; t.i[0] = t.i[1]; t.d[1] = t.d[2]; t.i[1] = t.i[2]; t.d[2] = INFINITY; t.i[2] = 0x7fffffff; }
            if (l == r) { rd = md; ri = mi; }
        }
        if (l < 3) {
            if (out_d) { out_d[3 * (size_t)q + l] = rd; out_i[3 * (size_t)q + l] = ri; }
            if (P.enabled) {
                const size_t e = 3 * (size_t)(P.q0 + q) + l;
                for (int g = 0; g < P.W.world; ++g) { scsh_c_dist(P.W, g)[e] = rd; scsh_c_idx(P.W, g)[e] = ri; }
            }
        }
    }
    if (P.enabled) scsh_raise(P.W, SCSH_C, *P.batch_p, P.counter);
}

}  // namespace liorf
