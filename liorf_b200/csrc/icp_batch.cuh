// icp_batch.cuh — loop-closure ICP for many keyframe pairs at once (liorf_loop_closure_icp_batch): per-pair target grids built in one
// pass, and one launch per ICP iteration / one for getFitnessScore covering every pair.  Each pair keeps exactly the block partition
// of the single-pair call (icp.cuh: blocks_p = min(ceil(n_src_p / 256), 4 SMs), grid-stride blocks_p * 256 within the pair, partials
// folded in block order by the pair's last block), so every result is bit-identical to liorf_loop_closure_icp on the same pair.
//
// Target grids: every pair gets the single-pair call's 256 x 256 x 32 torus of 1 m cells.  The iterations would be exact on any torus
// (a correspondence within max_corr_dist always ends the shell search by its break test), but getFitnessScore searches up to 64 shells
// and counts whatever it finds, so for a source point with no target point within 64 m the torus' aliasing decides the answer; a
// smaller torus per pair would change those fitness values.  The pairs' cell arrays are concatenated (pair q owns cells
// [q NC, (q + 1) NC)), so one count, one k_grid_scan and one scatter build all of them.
#pragma once
#include "icp.cuh"

namespace liorf {

struct IcpPairDesc {             // one pair of a wave that passed the size guards
    int src_off, n_src;          // its source cloud in the wave's voxel arrays
    int tgt_off, n_tgt;          // its target cloud there
    int tgt_first;               // first of its points in the concatenated cell-sorted target array
    int blocks, part_off;        // CTAs of the single-pair partition, first partial slot (in blocks)
    int pad;
};

__device__ __forceinline__ int icpb_pair_of_point(const IcpPairDesc* __restrict__ pd, int R, int i) {    // last pair with tgt_first <= i
    int lo = 0, hi = R - 1;
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (__ldg(&pd[mid].tgt_first) <= i) lo = mid; else hi = mid - 1; }
    return lo;
}

__global__ void __launch_bounds__(256) k_icpb_grid_count(const float4* __restrict__ vox, const IcpPairDesc* __restrict__ pd, int R, int total, GridDims g,
                                                         unsigned* __restrict__ counts) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int q = icpb_pair_of_point(pd, R, i);
    const float4 p = vox[pd[q].tgt_off + (i - pd[q].tgt_first)];
    atomicAdd(&counts[(size_t)q * grid_cells(g) + grid_cell_of(g, p.x, p.y, p.z)], 1u);
}
// fills each cell from its end (as k_grid_scatter); w = the point's index within ITS pair's target; counts return to zero
__global__ void __launch_bounds__(256) k_icpb_grid_scatter(const float4* __restrict__ vox, const IcpPairDesc* __restrict__ pd, int R, int total, GridDims g,
                                                           unsigned* __restrict__ counts, const unsigned* __restrict__ cell_start, float4* __restrict__ sorted) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int q = icpb_pair_of_point(pd, R, i);
    const int local = i - pd[q].tgt_first;
    const float4 p = vox[pd[q].tgt_off + local];
    const size_t c = (size_t)q * grid_cells(g) + grid_cell_of(g, p.x, p.y, p.z);
    const unsigned k = atomicSub(&counts[c], 1u) - 1u;
    sorted[cell_start[c] + k] = make_float4(p.x, p.y, p.z, __int_as_float(local));
}

// act[k] = (pair, first CTA of the pair in this launch), ascending in the CTA; CTAs of a pair that has finished return at once
__device__ __forceinline__ int icpb_slot_of_block(const int2* __restrict__ act, int n_act, int b) {
    int lo = 0, hi = n_act - 1;
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (__ldg(&act[mid].y) <= b) lo = mid; else hi = mid - 1; }
    return lo;
}

__global__ void __launch_bounds__(ICP_BLOCK) k_icpb_iteration(const IcpPairDesc* __restrict__ pd, const int2* __restrict__ act, int n_act, float4* __restrict__ src_cur,
                                                             IcpState* __restrict__ st, const unsigned* __restrict__ cell_start, const float4* __restrict__ gmap,
                                                             GridDims g, int r_max, float max_d2, double* __restrict__ partial, int* __restrict__ counters) {
    const int2 a = act[icpb_slot_of_block(act, n_act, (int)blockIdx.x)];
    const IcpPairDesc d = pd[a.x];
    icp_iteration_body(src_cur + d.src_off, d.n_src, st + a.x, cell_start + (size_t)a.x * grid_cells(g), gmap, g, r_max, max_d2,
                       partial + (size_t)d.part_off * ICP_NSUM, counters + a.x, nullptr, nullptr, nullptr, (int)blockIdx.x - a.y, d.blocks);
}

// getFitnessScore of every pair in act, with the final transformation each pair's loop left in its state; out[2 q .. 2 q + 1]
// (64 registers: left to itself ptxas picks 40 and spills the search state to the stack)
__global__ void __maxnreg__(64) k_icpb_fitness(const IcpPairDesc* __restrict__ pd, const int2* __restrict__ act, int n_act, const float4* __restrict__ src,
                                                           const IcpState* __restrict__ st, const unsigned* __restrict__ cell_start, const float4* __restrict__ gmap,
                                                           GridDims g, int r_max, double* __restrict__ partial, int* __restrict__ counters, double* __restrict__ out) {
    __shared__ float s_T[12];
    const int2 a = act[icpb_slot_of_block(act, n_act, (int)blockIdx.x)];
    const IcpPairDesc d = pd[a.x];
    if (threadIdx.x < 12) s_T[threadIdx.x] = st[a.x].final_T[threadIdx.x];
    __syncthreads();
    icp_fitness_body(src + d.src_off, d.n_src, s_T, cell_start + (size_t)a.x * grid_cells(g), gmap, g, r_max, partial + (size_t)d.part_off * 2,
                     counters + a.x, out + 2 * a.x, (int)blockIdx.x - a.y, d.blocks);
}

}  // namespace liorf
