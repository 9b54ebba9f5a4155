// sc_distance.cuh — stage 2 of detectLoopClosureID for query batches: distanceBtnScanContext (include/Scancontext.cpp:116-148)
// with the candidate descriptor staged by the TMA engine and the column / shift loops blocked in registers.
//
// One warp per (query, candidate) pair, looping over pairs.  The candidate's 20x60 fp64 descriptor (9 600 B, a random row of a database
// that lives in HBM) is fetched by ONE bulk asynchronous copy (cp.async.bulk → shared memory, completion on an mbarrier) while the warp
// derives the query's sector key / column norms and runs fastAlignUsingVkey.
// What bounds the kernel is not HBM but the SM's shared-memory port and fp64 pipe: a pair is ~32k fp64 operations (the reference's
// sequential, unfused sums) fed from shared memory.  Round 1 gave every lane two UNRELATED columns (l, l + 32) and two unrelated shifts:
// 15.6k 64-bit shared loads per pair, ~1 000 port cycles, and measured 1 570 cycles per pair per SM.  Here a lane owns two ADJACENT
// columns (2l, 2l+1) and two adjacent shifts:
//   fine search (:123-144)  the 7 shifts of 2 adjacent columns touch 8 consecutive candidate columns instead of 14 → 8 loads feed 14
//                           multiply-adds per ring; the query's two columns come as one 16-byte global load (two 8-byte loads for an 8-byte-aligned query array);
//   fastAlignUsingVkey (:93-113)  shift 2l+1 at column k reads what shift 2l read at column k-1 → carried in a register; the new value
//                           and the next one arrive as one 16-byte load, so do v1[k], v1[k+1] (broadcast);
// → ~7k shared loads (about 550 port cycles) per pair, same arithmetic in the same order: every fp64 sum keeps the reference's sequential
// order (k_sc_distance in scancontext.cuh, the straightforward form, stays in use for the live single-query call; results are
// bit-identical: tests/test_gpu_sc_tensor.py, test_gpu_deskew_sc.py, test_gpu_fullscale.py).
// Algorithmic traffic per pair: 9 600 B candidate + 9 600 B query descriptor (three pairs share a query: L2) + 960 B candidate keys/norms.
#pragma once
#include "sc_shard.cuh"

namespace liorf {

constexpr int SCDB_WARPS = 4;
constexpr int SCDB_THREADS = SCDB_WARPS * 32;
constexpr int SCDB_CHUNK = 5;                       // rings of the query descriptor per prefetch chunk of the fine search
constexpr int SCDB_VK1 = 64;                        // s_vk1 padded to 64 doubles (keeps the similarity buffer 16-byte aligned)
constexpr int SCDB_WARP_BYTES = SC_DESC * 8 + SCDB_VK1 * 8 + 7 * SC_SECTOR * 8;      // candidate descriptor + query sector key + 7 x 60 similarities = 13 472 B
constexpr int SCDB_SMEM = SCDB_WARPS * SCDB_WARP_BYTES + SCDB_WARPS * 8;
static_assert(SCDB_WARP_BYTES % 16 == 0, "per-warp shared-memory block must keep 16-byte alignment");

// Two adjacent columns of one ring of the caller's query descriptor.  kQ16: the descriptor array is 16-byte aligned → one 16-byte load;
// otherwise (a float64 tensor view at an odd element offset is only 8-byte aligned) two 8-byte loads of the same values.
template <bool kQ16>
__device__ __forceinline__ double2 scdb_query_pair(const double* p) {
    if constexpr (kQ16) return *reinterpret_cast<const double2*>(p);
    else return make_double2(p[0], p[1]);
}

// kQ16: qdesc is 16-byte aligned (sc_distance_launch picks the instantiation); both read the same values and compute bit-identical results
template <bool kQ16>
__global__ void __launch_bounds__(SCDB_THREADS, 4) k_sc_distance_bulk(const double* __restrict__ qdesc, const int* __restrict__ cand, int n_pairs, int cand_per_query,
                                                                  const double* __restrict__ db_desc, const double* __restrict__ db_sk, const double* __restrict__ db_cn,
                                                                  int own_begin, int own_count, double* __restrict__ out_dist, int* __restrict__ out_shift, int* err_flag,
                                                                  const int* __restrict__ pair_list, const int* __restrict__ n_list, ShardPush P) {
    extern __shared__ __align__(16) unsigned char scdb_smem[];
    const int w = warp_id(), l = lane_id();
    double* s_sc2 = reinterpret_cast<double*>(scdb_smem + (size_t)w * SCDB_WARP_BYTES);
    double* s_vk1 = s_sc2 + SC_DESC;
    double (*s_sim)[SC_SECTOR] = reinterpret_cast<double (*)[SC_SECTOR]>(s_vk1 + SCDB_VK1);
    const uint32_t bar = smem_u32(scdb_smem + (size_t)SCDB_WARPS * SCDB_WARP_BYTES + 8 * w);
    __shared__ int s_abort;
    if (threadIdx.x == 0) s_abort = 0;
    if (l == 0) mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();
    uint32_t parity = 0;
    const int n_warps = gridDim.x * SCDB_WARPS;
    const int n_items = pair_list ? *n_list : n_pairs;               // sharded search: the compact list of the pairs this rank owns
    const bool act = l < SC_SECTOR / 2;                              // 30 lanes own two adjacent columns / shifts each
    const int c0 = 2 * l;                                            // this lane's columns: c0, c0 + 1; its shifts: c0, c0 + 1
    for (int it = blockIdx.x * SCDB_WARPS + w; it < n_items; it += n_warps) {
        const int pair = pair_list ? pair_list[it] : it;
        const int q = pair / cand_per_query;
        const int c = cand[pair];
        if (c == 0x7fffffff || c < 0) { if (l == 0 && out_dist) { out_dist[pair] = INFINITY; out_shift[pair] = 0; } continue; }
        const int lc = c - own_begin;
        if (lc < 0 || lc >= own_count) continue;
        const double* sc1 = qdesc + (size_t)q * SC_DESC;
        __syncwarp();                                                   // every lane is done with the previous pair's buffers
        if (l == 0) { mbar_expect_tx(bar, SC_DESC * 8); bulk_g2s(smem_u32(s_sc2), db_desc + (size_t)lc * SC_DESC, SC_DESC * 8, bar); }
        // the candidate's sector key twice in a row (in the not yet used similarity buffer): circshift(vkey2, s)[k] = vk2d[k - s + 60]
        double* s_vk2d = &s_sim[0][0];
        // the QUERY's sector key and column norms are derived here, from the descriptor the fine search reads anyway (k_sc_keys_batch's
        // arithmetic: sequential sums over the rings, :214-227, :75-81) — no per-query key arrays, no kernel in front of this one
        double n1a = 0, n1b = 0;
        double2 qa[SCDB_CHUNK];                                       // the query's two columns, rings 0..4: kept for the fine search (see there)
        if (act) {
            double suma = 0, sqa = 0, sumb = 0, sqb = 0;
#pragma unroll
            for (int r = 0; r < SC_RING; ++r) {
                const double2 v = scdb_query_pair<kQ16>(sc1 + r * SC_SECTOR + c0);
                if (r < SCDB_CHUNK) qa[r] = v;
                suma += v.x; sqa += v.x * v.x; sumb += v.y; sqb += v.y * v.y;
            }
            *reinterpret_cast<double2*>(s_vk1 + c0) = make_double2(suma / SC_RING, sumb / SC_RING);
            n1a = sqrt(sqa); n1b = sqrt(sqb);
            const double2 v2 = *reinterpret_cast<const double2*>(db_sk + (size_t)lc * SC_SECTOR + c0);
            *reinterpret_cast<double2*>(s_vk2d + c0) = v2; *reinterpret_cast<double2*>(s_vk2d + SC_SECTOR + c0) = v2;
        }
        __syncwarp();
        // fastAlignUsingVkey (:93-113): lane ↔ shifts (c0, c0 + 1), sequential sum over the columns; first strict minimum of the norm.
        // A_k = vk2d[60 - c0 + k] belongs to shift c0 at column k and to shift c0 + 1 at column k + 1.
        double best = 10000000.0; int best_s = 0x7fffffff;
        if (act) {
            const double* pA = s_vk2d + SC_SECTOR - c0;              // even offset → 16-byte aligned pairs
            double carry = pA[-1];
            double ssA = 0, ssB = 0;
#pragma unroll 6
            for (int k = 0; k < SC_SECTOR; k += 2) {
                const double2 a = *reinterpret_cast<const double2*>(pA + k);
                const double2 v1 = *reinterpret_cast<const double2*>(s_vk1 + k);
                double dA = v1.x - a.x, dB = v1.x - carry;
                ssA += dA * dA; ssB += dB * dB;
                dA = v1.y - a.y; dB = v1.y - a.x;
                ssA += dA * dA; ssB += dB * dB;
                carry = a.y;
            }
            const double nA = sqrt(ssA), nB = sqrt(ssB);
            if (nA < best) { best = nA; best_s = c0; }               // ascending s within the lane ⇒ first minimum kept
            if (nB < best) { best = nB; best_s = c0 + 1; }
        }
        __syncwarp();                                                   // the similarity buffer is free again
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            double ob = __shfl_xor_sync(FULL, best, o); int os = __shfl_xor_sync(FULL, best_s, o);
            if (ob < best || (ob == best && os < best_s)) { best = ob; best_s = os; }
        }
        const int align = best_s == 0x7fffffff ? 0 : best_s;            // every norm >= 1e7 or NaN ⇒ argmin stays 0 (:95)
        // the 7 shifts {align-3 .. align+3} mod 60 in natural order m = 0..6; the reference visits them SORTED ascending (:123-130):
        // jpos[m] = rank of shift m in that order (they differ only when the window wraps around 0)
        int sh_m[7], jpos[7];
        {
            const int lo = SC_SEARCH_RADIUS - align;                    // > 0: the first `lo` shifts wrapped below 0 (→ 57..59) and sort LAST
            const int hi = align + SC_SEARCH_RADIUS - (SC_SECTOR - 1);  // > 0: the last `hi` shifts wrapped past 59 (→ 0..2) and sort FIRST
#pragma unroll
            for (int m = 0; m < 7; ++m) {
                int v = align + m - SC_SEARCH_RADIUS; v += v < 0 ? SC_SECTOR : 0; v -= v >= SC_SECTOR ? SC_SECTOR : 0;
                sh_m[m] = v;
                jpos[m] = lo > 0 ? (m < lo ? m + 7 - lo : m - lo) : hi > 0 ? (m >= 7 - hi ? m - (7 - hi) : m + hi) : m;
            }
        }
        // the candidate descriptor has landed (or the wait gives up with the error flag set)
        if (!mbar_wait(bar, parity, &s_abort, err_flag)) break;        // error flag is set; the epilogue below still runs (flags, counter)
        parity ^= 1u;
        // fine search (:123-144): lane ↔ query columns (c0, c0 + 1); for shift m column c0 meets candidate column c0 - sh_m = win[6 - m],
        // column c0 + 1 meets win[7 - m], win[i] = candidate column (c0 - align - 3 + i) mod 60: 8 consecutive columns for 14 dot products,
        // each summed over the 20 rings in ascending order
        if (act) {
            int idx[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) { int v = (c0 - align - SC_SEARCH_RADIUS + i) % SC_SECTOR; if (v < 0) v += SC_SECTOR; idx[i] = v; }
            double d0[7], d1[7];
#pragma unroll
            for (int m = 0; m < 7; ++m) { d0[m] = 0; d1[m] = 0; }
            // The query descriptor is NOT in shared memory (it would halve the pairs in flight) and, at 16 x 9.6 kB per SM, not in L1
            // either: a load issued where it is used waits a full L2 / HBM round trip (ncu r2: 40 % of this kernel's stall samples sat on
            // this loop).  So the rings arrive in chunks of SCDB_CHUNK, the NEXT chunk's loads in flight while this one is multiplied;
            // chunk 0 was kept from the key pass above.
#pragma unroll 1
            for (int ch = 0; ch < SC_RING / SCDB_CHUNK; ++ch) {
                double2 qb[SCDB_CHUNK];
                if (ch + 1 < SC_RING / SCDB_CHUNK) {
#pragma unroll
                    for (int u = 0; u < SCDB_CHUNK; ++u) qb[u] = scdb_query_pair<kQ16>(sc1 + ((ch + 1) * SCDB_CHUNK + u) * SC_SECTOR + c0);
                }
#pragma unroll
                for (int u = 0; u < SCDB_CHUNK; ++u) {
                    const double* row = s_sc2 + (ch * SCDB_CHUNK + u) * SC_SECTOR;
                    double win[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) win[i] = row[idx[i]];
#pragma unroll
                    for (int m = 0; m < 7; ++m) { d0[m] += qa[u].x * win[6 - m]; d1[m] += qa[u].y * win[7 - m]; }
                }
                if (ch + 1 < SC_RING / SCDB_CHUNK) {
#pragma unroll
                    for (int u = 0; u < SCDB_CHUNK; ++u) qa[u] = qb[u];
                }
            }
            const double* cn2 = db_cn + (size_t)lc * SC_SECTOR;
            double nw[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) nw[i] = cn2[idx[i]];
#pragma unroll
            for (int m = 0; m < 7; ++m) {
                const double n2a = nw[6 - m], n2b = nw[7 - m];
                const double sa = ((n1a == 0) | (n2a == 0)) ? -2.0 : d0[m] / (n1a * n2a);      // distDirectSC :73-88
                const double sb = ((n1b == 0) | (n2b == 0)) ? -2.0 : d1[m] / (n1b * n2b);
                *reinterpret_cast<double2*>(&s_sim[jpos[m]][c0]) = make_double2(sa, sb);
            }
        }
        __syncwarp();
        double dist = INFINITY; int sh = 0;
        if (l < 7) {
            double sum = 0; int eff = 0;
#pragma unroll 12
            for (int k = 0; k < SC_SECTOR; ++k) { double v = s_sim[l][k]; if (v != -2.0) { sum = sum + v; eff = eff + 1; } }     // the loads run ahead of the sequential adds
            dist = 1.0 - sum / eff;                                      // eff == 0 ⇒ NaN, never selected
#pragma unroll
            for (int m = 0; m < 7; ++m) if (jpos[m] == l) sh = sh_m[m];  // lane j holds the j-th smallest shift
        }
        double mn = 10000000.0; int arg = 0;
#pragma unroll
        for (int j = 0; j < 7; ++j) {
            double dj = __shfl_sync(FULL, dist, j); int sj = __shfl_sync(FULL, sh, j);
            if (dj < mn) { mn = dj; arg = sj; }
        }
        if (l == 0) {
            if (P.enabled) {             // push: entry [pair] of the pair array of every rank's window, straight from the warp that computed the pair
                for (int g = 0; g < P.W.world; ++g) { scsh_d_dist(P.W, g)[pair] = mn; scsh_d_shift(P.W, g)[pair] = arg; }
            } else { out_dist[pair] = mn; out_shift[pair] = arg; }
        }
    }
    if (P.enabled) scsh_raise(P.W, SCSH_D, *P.batch_p, P.counter);      // the last block to finish raises this rank's phase-D flag in every peer window
}

}  // namespace liorf
