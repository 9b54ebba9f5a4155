// prims.cuh — device-wide primitives written for sm_100a: single-pass exclusive scan with decoupled
// look-back, and a stable LSD radix sort of (u32 key, u32 value) pairs (one-sweep style: one global
// histogram kernel, then one kernel per 8-bit digit with per-digit look-back).
//
// Look-back status words carry an epoch so the status arrays are never memset between launches, and every
// spin is bounded: if a predecessor never shows up the kernel raises err_flag and bails out instead of hanging.
#pragma once
#include "common.cuh"

namespace liorf {

constexpr int SCAN_BLOCK = 256;
constexpr int SCAN_IPT = 8;
constexpr int SCAN_TILE = SCAN_BLOCK * SCAN_IPT;
constexpr unsigned SPIN_LIMIT = 1u << 24;

constexpr int SORT_BLOCK = 256;
constexpr int SORT_IPT = 8;
constexpr int SORT_TILE = SORT_BLOCK * SORT_IPT;
constexpr int SORT_WARPS = SORT_BLOCK / 32;
constexpr int RADIX_BITS = 8;
constexpr int RADIX = 1 << RADIX_BITS;

// status word: [63:34] epoch (30 bit) | [33:32] flag (1 = aggregate, 2 = inclusive prefix) | [31:0] value
__device__ __forceinline__ unsigned long long pack_status(unsigned epoch, unsigned flag, unsigned v) {
    return ((unsigned long long)(epoch & 0x3fffffffu) << 34) | ((unsigned long long)flag << 32) | v;
}
__device__ __forceinline__ unsigned long long ld_status(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ void st_status(unsigned long long* p, unsigned long long v) {
    asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Look-back for one chain (status index = tile * stride + chain), walked by ONE thread in batches of LB_BATCH
// predecessors whose loads are issued together (one L2 round trip per batch instead of per predecessor).
// Returns the exclusive prefix.
constexpr int LB_BATCH = 8;
__device__ __forceinline__ unsigned lookback_chain(unsigned long long* status, int tile, int stride, int chain, unsigned agg,
                                                   unsigned epoch, int* err_flag) {
    st_status(status + (size_t)tile * stride + chain, pack_status(epoch, tile == 0 ? 2u : 1u, agg));
    if (tile == 0) return 0u;
    const unsigned ep = epoch & 0x3fffffffu;
    unsigned excl = 0; unsigned spins = 0;
    int t = tile - 1;
    bool done = false;
    while (!done && t >= 0) {
        unsigned long long w[LB_BATCH];
#pragma unroll
        for (int j = 0; j < LB_BATCH; ++j) w[j] = (t - j >= 0) ? ld_status(status + (size_t)(t - j) * stride + chain) : pack_status(epoch, 2u, 0u);
        int used = 0;
#pragma unroll
        for (int j = 0; j < LB_BATCH; ++j) {
            if (done || used != j) continue;                      // stop at the first not-yet-published predecessor
            const unsigned flag = ((unsigned)(w[j] >> 34) == ep) ? (unsigned)((w[j] >> 32) & 3u) : 0u;
            if (flag == 0u) continue;
            excl += (unsigned)w[j]; ++used;
            if (flag == 2u) done = true;
        }
        t -= used;
        if (used == 0 && ++spins > SPIN_LIMIT) { atomicExch(err_flag, 1); return excl; }
    }
    st_status(status + (size_t)tile * stride + chain, pack_status(epoch, 2u, excl + agg));
    return excl;
}

// Warp-cooperative look-back for a single chain (stride 1): 32 lanes x 4 predecessors per step.
__device__ __forceinline__ unsigned lookback_warp(unsigned long long* status, int tile, unsigned agg, unsigned epoch, int* err_flag) {
    const int l = threadIdx.x & 31;
    if (l == 0) st_status(status + tile, pack_status(epoch, tile == 0 ? 2u : 1u, agg));
    if (tile == 0) return 0u;
    const unsigned ep = epoch & 0x3fffffffu;
    unsigned excl = 0; unsigned spins = 0;
    int t = tile - 1;                       // nearest predecessor not yet consumed
    while (t >= 0) {
        // lane l looks at predecessors t - (4 l + j); nearer ones have smaller offsets
        unsigned val[4]; unsigned flag[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int tt = t - (4 * l + j);
            unsigned long long w = tt >= 0 ? ld_status(status + tt) : pack_status(epoch, 2u, 0u);
            flag[j] = ((unsigned)(w >> 34) == ep) ? (unsigned)((w >> 32) & 3u) : 0u;
            val[j] = (unsigned)w;
        }
        // per lane: number of leading valid entries, whether a PREFIX ends the run, and the partial sum up to there
        unsigned cnt = 0, sum = 0; bool pre = false, open = true;
#pragma unroll
        for (int j = 0; j < 4; ++j) if (open) { if (flag[j] == 0u) open = false; else { sum += val[j]; ++cnt; if (flag[j] == 2u) { pre = true; open = false; } } }
        const unsigned full = __ballot_sync(FULL, cnt == 4u && !pre);        // lanes whose 4 entries are all aggregates
        const int first_stop = __ffs(~full) - 1;                             // first lane that is not "4 plain aggregates" (32 if none)
        const int fs = first_stop < 0 ? 32 : first_stop;
        unsigned contrib = (l < fs) ? sum : (l == fs ? sum : 0u);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) contrib += __shfl_xor_sync(FULL, contrib, o);
        const unsigned stop_cnt = __shfl_sync(FULL, cnt, fs < 32 ? fs : 0);
        const bool stop_pre = __shfl_sync(FULL, pre ? 1 : 0, fs < 32 ? fs : 0) != 0;
        excl += contrib;
        if (fs < 32) {
            if (stop_pre) { t = -1; break; }
            const int consumed = 4 * fs + (int)stop_cnt;
            t -= consumed;
            if (consumed == 0 && ++spins > SPIN_LIMIT) { if (l == 0) atomicExch(err_flag, 1); return excl; }
        } else t -= 128;
    }
    if (l == 0) st_status(status + tile, pack_status(epoch, 2u, excl + agg));
    return excl;
}

// Element count that is either known on the host or lives in device memory (so stages chain without host syncs).
// Grids are sized from `bound` (an upper bound known on the host).
struct Count {
    const int* dev; int host; int bound;
    __device__ __forceinline__ int get() const { return dev ? *dev : host; }
    static Count of_host(int n) { return Count{nullptr, n, n}; }
    static Count of_dev(const int* d, int bound) { return Count{d, 0, bound}; }
};

template <class T>
inline int reserve_zeroed(DevBuf<T>& b, size_t n, cudaStream_t s) {     // growth zero-fills (status arrays need a clean epoch)
    if (n <= b.cap) return LIORF_OK;
    int rc = b.reserve(n); if (rc) return rc;
    CUDA_TRY(cudaMemsetAsync(b.p, 0, b.cap * sizeof(T), s));
    return LIORF_OK;
}

// Ticket word of a look-back kernel: [63:32] launch epoch | [31:0] next tile ticket.  ONE atomicAdd hands a block its tile and
// the epoch that tags this launch's status words; the block that draws the last ticket stores (epoch + 1, 0) for the next
// launch.  Nothing about a launch is a host-side argument any more, so a chain of these kernels can be replayed from a CUDA graph.
constexpr unsigned long long TICKET_INIT = 1ull << 32;      // epoch 1: zero-filled status arrays (epoch 0) are never valid
__device__ __forceinline__ int draw_ticket(unsigned long long* ticket, unsigned& epoch) {
    const unsigned long long old = atomicAdd(ticket, 1ull);
    const int t = (int)(unsigned)(old & 0xffffffffull);
    epoch = (unsigned)(old >> 32);
    if (t == (int)gridDim.x - 1) atomicExch(ticket, (unsigned long long)(epoch + 1u) << 32);   // every ticket of this launch has been handed out
    return t;
}

struct ScanWork {            // per-scan scratch: ticket word + status array
    unsigned long long* ticket = nullptr;       // view: a word of the context's tickets, initialised to TICKET_INIT once
    DevBuf<unsigned long long> status;
    int* err_flag = nullptr;                    // view: the context's error flag
};

__device__ __forceinline__ unsigned warp_incl_scan(unsigned v) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { unsigned t = __shfl_up_sync(FULL, v, o); if (lane_id() >= o) v += t; }
    return v;
}

// Block-wide exclusive scan of per-thread totals; returns this thread's exclusive offset and the block total.
template <int BLOCK>
__device__ __forceinline__ unsigned block_excl_scan(unsigned v, unsigned* smem_warp /*BLOCK/32+1*/, unsigned& total) {
    unsigned incl = warp_incl_scan(v);
    if (lane_id() == 31) smem_warp[warp_id()] = incl;
    __syncthreads();
    if (warp_id() == 0) {
        unsigned w = lane_id() < BLOCK / 32 ? smem_warp[lane_id()] : 0u;
        unsigned wi = warp_incl_scan(w);
        if (lane_id() < BLOCK / 32) smem_warp[lane_id()] = wi - w;
        if (lane_id() == BLOCK / 32 - 1) smem_warp[BLOCK / 32] = wi;
    }
    __syncthreads();
    unsigned off = smem_warp[warp_id()] + incl - v;
    total = smem_warp[BLOCK / 32];
    __syncthreads();
    return off;
}

// Generic single-pass exclusive scan. LoadOp(i) -> unsigned value of element i; StoreOp(i, value, exclusive_prefix).
// total_out (optional) receives the grand total.
template <int BLOCK, int IPT, class LoadOp, class StoreOp>
__global__ void __launch_bounds__(BLOCK) k_scan_lookback(Count cnt, LoadOp load, StoreOp store, unsigned long long* ticket, unsigned long long* status,
                                                        int* err_flag, unsigned* total_out) {
    constexpr int SCAN_BLOCK = BLOCK, SCAN_IPT = IPT, SCAN_TILE = BLOCK * IPT;
    __shared__ int s_tile;
    __shared__ unsigned s_warp[SCAN_BLOCK / 32 + 1];
    __shared__ unsigned s_prefix;
    __shared__ unsigned s_epoch;
    const int n = cnt.get();
    const int ntiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    if (threadIdx.x == 0) { unsigned e; s_tile = draw_ticket(ticket, e); s_epoch = e; }
    __syncthreads();
    const int tile = s_tile;
    const unsigned epoch = s_epoch;
    if (tile >= ntiles) { if (n == 0 && tile == 0 && threadIdx.x == 0 && total_out) *total_out = 0u; return; }
    const int base = tile * SCAN_TILE + threadIdx.x * SCAN_IPT;
    unsigned v[SCAN_IPT]; unsigned sum = 0;
#pragma unroll
    for (int j = 0; j < SCAN_IPT; ++j) { int i = base + j; v[j] = i < n ? load(i) : 0u; sum += v[j]; }
    unsigned total;
    unsigned off = block_excl_scan<SCAN_BLOCK>(sum, s_warp, total);
    if (threadIdx.x < 32) { unsigned pf = lookback_warp(status, tile, total, epoch, err_flag); if (threadIdx.x == 0) s_prefix = pf; }
    __syncthreads();
    unsigned run = s_prefix + off;
#pragma unroll
    for (int j = 0; j < SCAN_IPT; ++j) { int i = base + j; if (i < n) store(i, v[j], run); run += v[j]; }
    if (total_out && tile == ntiles - 1 && threadIdx.x == SCAN_BLOCK - 1) *total_out = run;
}

template <int BLOCK = SCAN_BLOCK, int IPT = SCAN_IPT, class LoadOp, class StoreOp>
inline int launch_scan(Count n, LoadOp load, StoreOp store, ScanWork& w, unsigned* total_out, cudaStream_t s) {
    if (n.bound <= 0) { if (total_out) CUDA_TRY(cudaMemsetAsync(total_out, 0, sizeof(unsigned), s)); return LIORF_OK; }
    constexpr int TILE = BLOCK * IPT;
    int ntiles = (n.bound + TILE - 1) / TILE;
    int rc = reserve_zeroed(w.status, ntiles, s); if (rc) return rc;
    k_scan_lookback<BLOCK, IPT><<<ntiles, BLOCK, 0, s>>>(n, load, store, w.ticket, w.status.p, w.err_flag, total_out);
    CUDA_TRY(cudaGetLastError());
    return LIORF_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Radix sort
// ---------------------------------------------------------------------------------------------------------------
// global histograms of all four digits in one pass; hist layout [pass][256]
__global__ void __launch_bounds__(256) k_radix_hist(const unsigned* __restrict__ keys, Count cnt, unsigned* __restrict__ hist) {
    __shared__ unsigned sh[4 * RADIX];
    const int n = cnt.get();
    for (int i = threadIdx.x; i < 4 * RADIX; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        unsigned k = keys[i];
        atomicAdd(&sh[k & 255u], 1u); atomicAdd(&sh[RADIX + ((k >> 8) & 255u)], 1u);
        atomicAdd(&sh[2 * RADIX + ((k >> 16) & 255u)], 1u); atomicAdd(&sh[3 * RADIX + (k >> 24)], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 4 * RADIX; i += blockDim.x) if (sh[i]) atomicAdd(&hist[i], sh[i]);
}

// One stable counting pass on digit `shift`.  vals_in == nullptr means value = element index (first pass).
__global__ void __launch_bounds__(SORT_BLOCK) k_radix_pass(const unsigned* __restrict__ keys_in, const unsigned* __restrict__ vals_in,
                                                           unsigned* __restrict__ keys_out, unsigned* __restrict__ vals_out, Count cnt, int shift,
                                                           const unsigned* __restrict__ ghist /*256 counts of this digit*/, unsigned long long* ticket,
                                                           unsigned long long* status, int* err_flag) {
    __shared__ int s_tile;
    __shared__ unsigned s_epoch;
    __shared__ unsigned s_whist[SORT_WARPS][RADIX];   // per-warp digit counts → exclusive warp offsets
    __shared__ unsigned s_base[RADIX];                // global base + tile exclusive prefix per digit
    __shared__ unsigned s_warp[SORT_BLOCK / 32 + 1];
    const int n = cnt.get();
    const int ntiles = (n + SORT_TILE - 1) / SORT_TILE;
    if (threadIdx.x == 0) { unsigned e; s_tile = draw_ticket(ticket, e); s_epoch = e; }
    for (int i = threadIdx.x; i < SORT_WARPS * RADIX; i += SORT_BLOCK) (&s_whist[0][0])[i] = 0;
    __syncthreads();
    const int tile = s_tile;
    const unsigned epoch = s_epoch;
    if (tile >= ntiles) return;
    const int w = warp_id(), l = lane_id();
    const int wbase = tile * SORT_TILE + w * (32 * SORT_IPT);
    unsigned key[SORT_IPT], val[SORT_IPT], rank[SORT_IPT];
    const unsigned lt_mask = (1u << l) - 1u;
#pragma unroll
    for (int j = 0; j < SORT_IPT; ++j) {
        int i = wbase + j * 32 + l;
        bool valid = i < n;
        key[j] = valid ? keys_in[i] : 0xffffffffu;
        val[j] = valid ? (vals_in ? vals_in[i] : (unsigned)i) : 0u;
        unsigned d = (key[j] >> shift) & (RADIX - 1);
        unsigned vm = __ballot_sync(FULL, valid);
        unsigned mm = __match_any_sync(FULL, d) & vm;
        unsigned old = 0;
        int leader = __ffs(mm) - 1;
        if (valid && l == leader) { old = s_whist[w][d]; s_whist[w][d] = old + __popc(mm); }
        __syncwarp();
        old = __shfl_sync(FULL, old, leader < 0 ? 0 : leader);
        rank[j] = old + __popc(mm & lt_mask);
    }
    __syncthreads();
    // thread d: exclusive scan over warps of digit d, tile total, look-back, global base
    {
        const int d = threadIdx.x;      // SORT_BLOCK == RADIX
        unsigned run = 0;
#pragma unroll
        for (int ww = 0; ww < SORT_WARPS; ++ww) { unsigned c = s_whist[ww][d]; s_whist[ww][d] = run; run += c; }
        unsigned excl = lookback_chain(status, tile, RADIX, d, run, epoch, err_flag);
        // exclusive scan of the global digit histogram (each block redundantly; 256 values)
        unsigned g = ghist[d]; unsigned total;
        unsigned goff = block_excl_scan<SORT_BLOCK>(g, s_warp, total);
        s_base[d] = goff + excl;
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < SORT_IPT; ++j) {
        int i = wbase + j * 32 + l;
        if (i < n) {
            unsigned d = (key[j] >> shift) & (RADIX - 1);
            unsigned pos = s_base[d] + s_whist[w][d] + rank[j];
            keys_out[pos] = key[j]; vals_out[pos] = val[j];
        }
    }
}

struct SortWork {
    DevBuf<unsigned> keys_alt, vals_a, vals_b, hist;
    DevBuf<unsigned long long> status;
    unsigned long long* ticket = nullptr;       // view: a word of the context's tickets, initialised to TICKET_INIT once (see draw_ticket)
    int* err_flag = nullptr;                    // view: the context's error flag
};

// Sorts keys (in place semantic: result ends in keys / vals_out) stably; values start as iota.
// After 4 passes the result is back in the original `keys` buffer and in work.vals_b.
inline int radix_sort_pairs_iota(unsigned* keys, Count cnt, SortWork& w, unsigned** sorted_vals, cudaStream_t s) {
    *sorted_vals = nullptr;
    const int n = cnt.bound;
    if (n <= 0) return LIORF_OK;
    int rc;
    if ((rc = w.keys_alt.reserve(n))) return rc;
    if ((rc = w.vals_a.reserve(n))) return rc;
    if ((rc = w.vals_b.reserve(n))) return rc;
    if ((rc = w.hist.reserve(4 * RADIX))) return rc;
    int ntiles = (n + SORT_TILE - 1) / SORT_TILE;
    if ((rc = reserve_zeroed(w.status, (size_t)ntiles * RADIX, s))) return rc;
    CUDA_TRY(cudaMemsetAsync(w.hist.p, 0, 4 * RADIX * sizeof(unsigned), s));
    int hb = (n + 256 * 16 - 1) / (256 * 16); if (hb > 4 * kNumSMs) hb = 4 * kNumSMs; if (hb < 1) hb = 1;
    k_radix_hist<<<hb, 256, 0, s>>>(keys, cnt, w.hist.p);
    unsigned* kin = keys; unsigned* kout = w.keys_alt.p;
    unsigned* vin = nullptr; unsigned* vout = w.vals_a.p;
    for (int p = 0; p < 4; ++p) {
        k_radix_pass<<<ntiles, SORT_BLOCK, 0, s>>>(kin, vin, kout, vout, cnt, 8 * p, w.hist.p + p * RADIX, w.ticket, w.status.p, w.err_flag);
        unsigned* t = kin; kin = kout; kout = t;
        vin = vout; vout = (vin == w.vals_a.p) ? w.vals_b.p : w.vals_a.p;
    }
    CUDA_TRY(cudaGetLastError());
    // after 4 passes: keys back in `keys`, values in vals_b
    *sorted_vals = vin;
    return LIORF_OK;
}

}  // namespace liorf
