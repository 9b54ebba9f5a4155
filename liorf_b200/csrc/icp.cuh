// icp.cuh — the registration that consumes detectLoopClosureID's answer: performSCLoopClosure's
// pcl::IterativeClosestPoint (src/mapOptmization.cpp:652-674) on the GPU (SURVEY §8f row 3).
//   correspondence estimation : exact nearest neighbour of every source point in the target cloud, FLANN L2_Simple
//                               arithmetic (((dx*dx) + dy*dy) + dz*dz, fp32, no FMA), ties by original index; the
//                               target lives in the same 1 m voxel-hash grid the scan-to-map solver uses and the search
//                               grows cube shells until no unvisited cell can hold a closer point
//   transformation estimation : the 17 sums the SVD step needs (count, sum s, sum d, sum d s^T, sum d2) reduced in fp64 by
//                               a fixed tree + last-block fold (no float atomics: bit-reproducible)
// The 3x3 SVD / convergence logic is the scalar code of host/host_logic.hpp (as in PCL), run by the LAST block of every iteration on the
// device: the loop state (incremental and accumulated transform, convergence criteria) lives in device memory, an iteration that
// finds the loop finished returns at once, and the host reads the state back once per chunk of iterations instead of once per iteration.
#pragma once
#include "localmap.cuh"
#include "../host/host_logic.hpp"

namespace liorf {

constexpr int ICP_NSUM = 17;      // n, sx sy sz, dx dy dz, H[3][3] (H[r][c] = sum d_r s_c), sum of squared distances
constexpr int ICP_BLOCK = 256;

struct IcpT { float t[12]; };     // row-major 3x4, passed by value
struct IcpState {                 // device-resident loop state of pcl::IterativeClosestPoint::computeTransformation
    float inc[16];                // transformation_ of the last iteration (applied to the source at the start of the next)
    float final_T[16];            // final_transformation_
    liorf_host::IcpConvergence cc;
    int iterations, done, converged, pad;
};

__device__ __forceinline__ void icp_visit(const unsigned* __restrict__ cell_start, const float4* __restrict__ gmap, GridDims g, int x, int y, int z,
                                          const float4 q, float& bd, int& bi, float4& bp) {
    const int c = ((z & (g.DZ - 1)) * g.DY + (y & (g.DY - 1))) * g.DX + (x & (g.DX - 1));
    const unsigned b = __ldg(cell_start + c), e = __ldg(cell_start + c + 1);
    for (unsigned k = b; k < e; ++k) {
        const float4 p = __ldg(gmap + k);
        const float dx = q.x - p.x, dy = q.y - p.y, dz = q.z - p.z;
        float d = dx * dx; d += dy * dy; d += dz * dz;
        const int oi = __float_as_int(p.w);
        if (d < bd || (d == bd && oi < bi)) { bd = d; bi = oi; bp = p; }
    }
}

// exact nearest neighbour; the search stops after shell r once the best squared distance is below r^2 (every unvisited
// point is at least r away), or at r_max.  Returns false when the target is empty within r_max shells.
__device__ __forceinline__ bool icp_nearest(const float4 q, const unsigned* __restrict__ cell_start, const float4* __restrict__ gmap, GridDims g, int r_max,
                                            float& bd, int& bi, float4& bp) {
    const int cx = (int)floorf(q.x), cy = (int)floorf(q.y), cz = (int)floorf(q.z);
    bd = INFINITY; bi = 0x7fffffff; bp = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int r = 0; r <= r_max; ++r) {
        for (int dz = -r; dz <= r; ++dz)
            for (int dy = -r; dy <= r; ++dy) {
                const bool face = (dz == -r || dz == r || dy == -r || dy == r);
                if (face) { for (int dx = -r; dx <= r; ++dx) icp_visit(cell_start, gmap, g, cx + dx, cy + dy, cz + dz, q, bd, bi, bp); }
                else { icp_visit(cell_start, gmap, g, cx - r, cy + dy, cz + dz, q, bd, bi, bp); icp_visit(cell_start, gmap, g, cx + r, cy + dy, cz + dz, q, bd, bi, bp); }
            }
        if (bd < (float)r * (float)r) break;
    }
    return bi != 0x7fffffff;
}

// One ICP iteration's device half for ONE cloud pair, run by block `blk` of the `nblk` blocks that pair owns.  src_cur ← T_inc * src_cur
// (pcl::transformPointCloud with the previous iteration's estimate; identity on the first), correspondences with squared distance
// <= max_d2, per-block partial sums folded in block order by the pair's last block, which then runs the estimate / convergence step.
// The block partition (blk, nblk, grid-stride nblk * ICP_BLOCK) is the whole of what fixes the fp64 summation order, so the single-pair
// kernel and the batched one (icp_batch.cuh) give bit-identical results for the same pair.
// out (nullable): the folded sums.  nn_idx / nn_d2 (nullable): the neighbour index / squared distance per source point (tests).
__device__ __forceinline__ void icp_iteration_body(float4* __restrict__ src_cur, int n_src, IcpState* __restrict__ st, const unsigned* __restrict__ cell_start,
                                                   const float4* __restrict__ gmap, GridDims g, int r_max, float max_d2, double* __restrict__ partial,
                                                   int* __restrict__ counter, double* __restrict__ out, int* __restrict__ nn_idx, float* __restrict__ nn_d2,
                                                   int blk, int nblk) {
    __shared__ double s_red[ICP_BLOCK / 32][ICP_NSUM];
    __shared__ bool s_last;
    __shared__ float s_T[12];
    __shared__ double s_out[ICP_NSUM];
    if (__ldcg(&st->done)) return;                             // the loop ended in an earlier launch of this chunk
    if (threadIdx.x < 12) s_T[threadIdx.x] = __ldcg(&st->inc[threadIdx.x]);        // (rewritten only by this launch's LAST block, after every block has read it)
    __syncthreads();
    double acc[ICP_NSUM];
#pragma unroll
    for (int k = 0; k < ICP_NSUM; ++k) acc[k] = 0.0;
    for (int i = blk * ICP_BLOCK + threadIdx.x; i < n_src; i += nblk * ICP_BLOCK) {
        const float4 p = apply_affine_dev(s_T, src_cur[i]);
        src_cur[i] = p;
        float bd; int bi; float4 bp;
        const bool found = icp_nearest(p, cell_start, gmap, g, r_max, bd, bi, bp) && bd <= max_d2;
        if (nn_idx) { nn_idx[i] = found ? bi : -1; nn_d2[i] = bd; }
        if (found) {
            const double sx = p.x, sy = p.y, sz = p.z, dx = bp.x, dy = bp.y, dz = bp.z;
            acc[0] += 1.0; acc[1] += sx; acc[2] += sy; acc[3] += sz; acc[4] += dx; acc[5] += dy; acc[6] += dz;
            acc[7] += dx * sx; acc[8] += dx * sy; acc[9] += dx * sz; acc[10] += dy * sx; acc[11] += dy * sy; acc[12] += dy * sz;
            acc[13] += dz * sx; acc[14] += dz * sy; acc[15] += dz * sz; acc[16] += (double)bd;
        }
    }
#pragma unroll
    for (int k = 0; k < ICP_NSUM; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(FULL, acc[k], o);
    }
    if (lane_id() == 0) for (int k = 0; k < ICP_NSUM; ++k) s_red[warp_id()][k] = acc[k];
    __syncthreads();
    if (threadIdx.x < ICP_NSUM) {
        double s = 0; for (int w = 0; w < ICP_BLOCK / 32; ++w) s += s_red[w][threadIdx.x];
        partial[blk * ICP_NSUM + threadIdx.x] = s;
        __threadfence();
    }
    __syncthreads();
    if (threadIdx.x == 0) { const int t = atomicAdd(counter, 1); s_last = (t == nblk - 1); }
    __syncthreads();
    if (!s_last) return;
    if (threadIdx.x < ICP_NSUM) {                              // fold the per-block partials in block order (deterministic whoever is last)
        const volatile double* vp = partial;
        double s = 0; for (int b = 0; b < nblk; ++b) s += vp[b * ICP_NSUM + threadIdx.x];
        if (out) out[threadIdx.x] = s;
        s_out[threadIdx.x] = s;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        *counter = 0;
        // transformation estimation + convergence criteria (pcl::IterativeClosestPoint::computeTransformation's loop body, :652-674)
        float inc[16], fin[16];
        if (!liorf_host::icp_estimate(s_out, inc)) { st->cc.state = liorf_host::IcpConvergence::NO_CORRESPONDENCES; st->converged = 0; st->done = 1; }
        else {
            for (int k = 0; k < 16; ++k) fin[k] = st->final_T[k];
            liorf_host::mat4_mul(inc, fin, fin);                  // final_transformation_ = transformation_ * final_transformation_
            for (int k = 0; k < 16; ++k) { st->final_T[k] = fin[k]; st->inc[k] = inc[k]; }
            st->iterations += 1;
            liorf_host::IcpConvergence cc = st->cc;
            if (cc.has_converged(inc, s_out[16] / s_out[0])) { st->converged = 1; st->done = 1; }
            st->cc = cc;
        }
        __threadfence();
    }
}

__global__ void __launch_bounds__(ICP_BLOCK) k_icp_iteration(float4* __restrict__ src_cur, int n_src, IcpState* __restrict__ st, const unsigned* __restrict__ cell_start,
                                                            const float4* __restrict__ gmap, GridDims g, int r_max, float max_d2, double* __restrict__ partial,
                                                            int* __restrict__ counter, double* __restrict__ out, int* __restrict__ nn_idx, float* __restrict__ nn_d2) {
    icp_iteration_body(src_cur, n_src, st, cell_start, gmap, g, r_max, max_d2, partial, counter, out, nn_idx, nn_d2, (int)blockIdx.x, (int)gridDim.x);
}

// getFitnessScore (pcl::Registration::getFitnessScore, max_range = DBL_MAX) for ONE pair, block `blk` of its `nblk`: mean squared
// nearest-neighbour distance of the ORIGINAL source transformed by the final transformation T (row-major 3x4).  out[0] = sum d2, out[1] = count.
__device__ __forceinline__ void icp_fitness_body(const float4* __restrict__ src, int n_src, const float* T, const unsigned* __restrict__ cell_start,
                                                 const float4* __restrict__ gmap, GridDims g, int r_max, double* __restrict__ partial,
                                                 int* __restrict__ counter, double* __restrict__ out, int blk, int nblk) {
    __shared__ double s_red[ICP_BLOCK / 32][2];
    __shared__ bool s_last;
    double sum = 0.0, cnt = 0.0;
    for (int i = blk * ICP_BLOCK + threadIdx.x; i < n_src; i += nblk * ICP_BLOCK) {
        const float4 p = apply_affine_dev(T, src[i]);
        float bd; int bi; float4 bp;
        if (icp_nearest(p, cell_start, gmap, g, r_max, bd, bi, bp)) { sum += (double)bd; cnt += 1.0; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { sum += __shfl_xor_sync(FULL, sum, o); cnt += __shfl_xor_sync(FULL, cnt, o); }
    if (lane_id() == 0) { s_red[warp_id()][0] = sum; s_red[warp_id()][1] = cnt; }
    __syncthreads();
    if (threadIdx.x < 2) {
        double s = 0; for (int w = 0; w < ICP_BLOCK / 32; ++w) s += s_red[w][threadIdx.x];
        partial[blk * 2 + threadIdx.x] = s;
        __threadfence();
    }
    __syncthreads();
    if (threadIdx.x == 0) { const int t = atomicAdd(counter, 1); s_last = (t == nblk - 1); }
    __syncthreads();
    if (!s_last) return;
    if (threadIdx.x < 2) {
        const volatile double* vp = partial;
        double s = 0; for (int b = 0; b < nblk; ++b) s += vp[b * 2 + threadIdx.x];
        out[threadIdx.x] = s;
    }
    if (threadIdx.x == 0) *counter = 0;
}

__global__ void __launch_bounds__(ICP_BLOCK) k_icp_fitness(const float4* __restrict__ src, int n_src, IcpT T_final, const unsigned* __restrict__ cell_start,
                                                          const float4* __restrict__ gmap, GridDims g, int r_max, double* __restrict__ partial,
                                                          int* __restrict__ counter, double* __restrict__ out) {
    icp_fitness_body(src, n_src, T_final.t, cell_start, gmap, g, r_max, partial, counter, out, (int)blockIdx.x, (int)gridDim.x);
}

}  // namespace liorf
