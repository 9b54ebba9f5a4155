// capi.cu — context + extern "C" entry points declared in include/liorf_b200.h.
// One translation unit; every kernel lives in the .cuh files next to this one.  Built with
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -fmad=false
#include <map>
#include <algorithm>
#include "../../include/liorf_b200.h"
#include "common.cuh"
#include "prims.cuh"
#include "voxelgrid.cuh"
#include "localmap.cuh"
#include "scan2map.cuh"
#include "deskew.cuh"
#include "scancontext.cuh"
#include "sc_tensor.cuh"
#include "sc_shard.cuh"
#include "sc_distance.cuh"
#include "icp.cuh"
#include "icp_batch.cuh"
#include "../host/host_logic.hpp"
#include <vector>
#include <cstring>
#include <cmath>
#include <new>
#include <chrono>
#include <cstdlib>

using namespace liorf;

// NVTX range around every C-ABI entry that touches the device (SURVEY §5: "NVTX ranges per hot-path function"): nsys / ncu --nvtx show the
// reference's function boundaries (projectPointCloud, downsampleCurrentScan, scan2MapOptimization ...) on the timeline.  Header-only NVTX v3:
// without a profiler attached a push/pop pair is two predicted branches.
#include <nvtx3/nvToolsExt.h>
struct NvtxRange { explicit NvtxRange(const char* name) { nvtxRangePushA(name); } ~NvtxRange() { nvtxRangePop(); } };
#define LIORF_NVTX NvtxRange nvtx_range_(__func__)

static_assert(sizeof(S2MTrace) == sizeof(liorf_lm_trace), "trace layout mismatch");
static_assert(sizeof(liorf_point_xyzirt) == sizeof(RawPoint), "raw point layout mismatch");
static_assert(S2M_MAX_ITERS == LIORF_MAX_ITERS, "iteration cap mismatch");

enum { C_N_SCAN = 0, C_N_DS, C_M_DS, C_NSEL, C_FIRST_KEPT, C_CONV, C_HOOK_NSEL, C_COUNT = 16 };

struct Keyframe { size_t off; int count; float pose[6]; double time; };

// optional per-section CUDA-event timing on the context's stream (bench.py's live roofline numbers)
enum { SEC_DESKEW = 0, SEC_DOWNSAMPLE, SEC_MAP_BUILD, SEC_GRID_BUILD, SEC_SCAN2MAP, SEC_SC_MAKE, SEC_SC_SEARCH, SEC_SC_GEMM, SEC_COUNT = 8 };
constexpr int PROF_RING = 64;
constexpr int S2M_SPARE_SMS = 16;      // SMs the persistent solver leaves to the concurrent front end of the next frame
struct Profiler {
    bool enabled = false; unsigned mask = 0xffu;        // mask: sections that record events (bit = section id)
    Event ev[PROF_RING][2]; int sec[PROF_RING]; int pending = 0; bool created = false;
    double ms[SEC_COUNT] = {0}; long long calls[SEC_COUNT] = {0};
};

// The ScanContext database: one context owns it, others may borrow it (liorf_sc_borrow_database)
struct ScDatabase { DevBuf<double> desc, sk, cn; DevBuf<float> keys; };

// Every member that holds a CUDA resource owns it (common.cuh); raw pointers are views into memory another member owns.
struct liorf_ctx {
    liorf_params P;
    Stream stream;
    int num_sms = kNumSMs;
    // device scalars
    int* d_counts = nullptr;        // view: C_COUNT ints of the CURRENT front set (N_SCAN, N_DS, FIRST_KEPT, hook counts)
    DevMem<int> d_counts_base;      // [front set 0 | shared | front set 1], C_COUNT ints each: either set is contiguous with the shared block
    int* d_shared = nullptr;        // view: counts that do not belong to a front set (C_M_DS)
    DevMem<int> d_misc;             // counters / error flag (zero-initialised)
    DevMem<unsigned long long> d_tick;   // look-back ticket words (prims.cuh: draw_ticket), one per scan / sort work area
    int* d_err = nullptr;           // view: d_misc[0]
    HostBuf<int> h_mail;            // pinned mailbox (128 KB: scalars/trace in the lower half, IMU table staging in the upper)
    // clouds
    DevBuf<float4> scan, scan_ds, map_raw, map_ds, kf_points;
    DevBuf<int> membership, out_keys;
    int n_scan_bound = 0;           // host-known upper bound of laserCloudSurfLast / DS counts
    int h_n_scan = -1, h_n_ds = -1, h_m_ds = -1;   // host copies (-1 = unknown)
    int rep_counts[3] = {-1, -1, -1};              // n_scan, n_ds, m_ds as of the last pose read-back (liorf_get_last_counts)
    int m_bound = 0;
    VoxelGridWork vg;               // scan-side VoxelGrid work area (main stream)
    VoxelGridWork vg_map;           // map-side work area: the local-map chain runs concurrently on stream_map
    Stream stream_map;
    Event ev_main, ev_map; bool map_pending = false;
    MapGrid grid;
    DeskewWork dk;
    std::vector<Keyframe> kfs;
    size_t kf_used = 0;
    DevBuf<KfSel> d_sel;
    HostBuf<KfSel> h_sel;                            // two halves, alternated per call (see stage_slot)
    Event stage_ev[2][2]; int stage_turn[2] = {0, 0};   // [0] = selection table, [1] = IMU table
    // the local-map chain as CUDA graphs (one pair per 64k-point size bucket): ~20 stream operations become 2 launches
    struct MapGraphs { GraphExec vg, grid; const void* sig[20] = {nullptr}; };
    std::map<int, MapGraphs> map_graphs; bool use_graphs = true;
    std::vector<int> last_sel; unsigned long long pose_version = 0, last_sel_version = ~0ull; bool map_valid = false;
    // LM
    DevMem<float> d_tf6; DevMem<LMDeviceState> d_lm; DevMem<S2MTrace> d_trace; DevMem<double> d_partial; DevMem<ulonglong2> d_wpart; DevMem<unsigned long long> d_res; DevMem<long long> d_dbg; DevMem<unsigned long long> d_dbg_gt;
    DevMem<IcpState> icp_state; DevBuf<QueryCache> qcache; DevBuf<float4> cand; unsigned s2m_launch_seq = 0; DevMem<S2MMail> d_mail; bool mail_fresh = false; bool s2m_global_state = false;
    int s2m_grid = 0; bool s2m_no_cache = false; int map_vg_grid = 0;
    int s2m_ctas = 0;                // tests: solver CTAs of every launch (0 = num_sms per function call, s2m_grid in liorf_process_frame)
    int vg_ctas = 0;                 // tests: CTAs of liorf_voxel_grid's one-kernel VoxelGrid (0 = num_sms)
    DevBuf<float4> h_coeff, h_sel_pts, h_ori_c, h_coeff_c; DevBuf<unsigned char> h_flag; DevBuf<int> h_idx; DevBuf<float> h_d2, h_plane;
    DevBuf<double> lm_partial; ScanWork combine_scan; int hook_n = 0;
    DevMem<float> d_lm_out;         // AtA[36] AtB[6] X[6]
    // ScanContext
    ScDatabase sc_own; ScDatabase* sc_db = &sc_own; int sc_n = 0;   // sc_db: sc_own, or the owner's database when borrowed
    bool sc_borrowed() const { return sc_db != &sc_own; }
    DevMem<unsigned> d_bins;
    int sc_tree_n = 0, sc_counter = 0;
    DevBuf<float> sc_part_d; DevBuf<int> sc_part_i;
    DevBuf<float> sc_q_d; DevBuf<int> sc_q_i; DevBuf<double> sc_pair_d; DevBuf<int> sc_pair_s;
    DevBuf<double> sc_qdesc; DevBuf<float> sc_qkeys; DevBuf<int> sc_res_i; DevBuf<double> sc_res_d;
    // batched detectLoopClosureID: answers + query indices in one device block (one download, one upload) and its pinned host mirror
    DevBuf<int> scdb_io; HostBuf<int> h_scdb;
    // tensor-core ring-key search (sc_tensor.cuh): operand images + work buffers.  A KeySet = a ring-key array the filter searches + the B
    // operand image built from it: ks_local = this context's own rows (sc_db->keys), ks_all = the replicated index of a sharded database
    struct KeySet { const float* keys = nullptr; int n = 0; unsigned gen = 0; DevBuf<uint8_t> bimg; DevMem<float> center; DevMem<unsigned> nmax;   // keys: view
                    int img_n = -1; unsigned img_gen = 0; const float* img_keys = nullptr; } ks_local, ks_all;
    DevBuf<uint8_t> sct_aimg; DevBuf<float> sct_cmin, sct_cmin32, sct_qnorm, sct_part; DevBuf<int> sct_cand, sct_cnt;
    DevMem<int> sct_over_cnt;
    // loop-closure ICP (icp.cuh)
    DevBuf<float4> icp_raw, icp_src, icp_src0, icp_tgt; MapGrid icp_grid; DevBuf<double> icp_partial; DevMem<double> icp_out; int* icp_counter = nullptr;   // icp_counter: view
    DevBuf<KfSel> icp_sel; DevBuf<int> icp_nn_idx; DevBuf<float> icp_nn_d2;
    // batched loop-closure ICP (icp_batch.cuh): work buffers of its own, sized by the largest wave so far
    struct IcpBatch {
        DevBuf<KfSel> sel; DevBuf<VgSegTile> tiles; DevBuf<int> seg_n, seg_vox, counters; DevBuf<unsigned> mm, keys, seg_start, counts, cell_start;
        DevBuf<VoxMeta> metas; DevBuf<unsigned long long> seg_base; DevBuf<float4> raw, vox, src_cur, sorted;
        DevBuf<IcpPairDesc> pd; DevBuf<int2> act; DevBuf<IcpState> st; DevBuf<double> partial, fit;
        SortWork sort; ScanWork scan, grid_scan;
        DevMem<int> d_flags;                    // [0] voxel total of the wave, [1] key range beyond 32 bits
        HostBuf<unsigned char> h_stage;         // pinned: tables going up, counts / states / sums coming back
        int max_pairs = 0;                      // tests: pairs per wave (0 = memory-bounded)
    } icpb;
    liorf_guess_state guess_state = {}; float tf_mapped[6] = {0, 0, 0, 0, 0, 0};   // updateInitialGuess statics + transformTobeMapped
    // sharded search over peer windows (sc_shard.cuh)
    // W.base[] and W.keys_all[] are views: of win, of a peer's window mapped into ipc[], or of a window of another context in this process
    struct ScShard { bool ready = false; ShardWin W; int qmax = 0, kcap = 0; size_t win_bytes = 0, off_keys = 0; unsigned* d_batch = nullptr; DevMem<unsigned> d_counter;
                     DevMem<unsigned char> win; IpcMapping<unsigned char> ipc[SCSH_MAX]; unsigned keys_gen = 0; bool keys_pushed = false;
                     GraphExec graph; const void* gsig[40] = {nullptr}; const void* last_sig[40] = {nullptr};
                     DevBuf<int> list; int* d_nlist = nullptr; } shard;   // d_batch, d_nlist, W.wait_ns: views of d_counter
    int sc_path = 0;                 // 0 auto, 1 CUDA-core brute force, 2 tensor-core filter + exact re-rank
    bool sct_attr_set = false; int sct_last_Q = 0; bool scdb_attr_set = false; int scdb_blocks_per_sm[2] = {1, 1};   // [kQ16]
    Profiler prof;
    double host_us[12] = {0}; long long host_frames = 0; bool host_timing = false;   // LIORF_HOST_TIMING=1 ([6..10]: pieces of the keyframe tail)
    Event tl_ev[8]; double tl_ms[8] = {0}; // debug GPU timeline stamps of process_frame
    long long launches = 0;         // kernels launched by this context (bench.py's gpu_launches)
    // ---- pipelined front end (cloudHandler of frame i+1 overlaps laserCloudInfoHandler of frame i) ----
    // Everything projectPointCloud + downsampleCurrentScan read or write for ONE frame lives in a "front set"; the context
    // holds two and swaps them, so the next frame's set is filled on stream_pre while the solver works on the current one.
    struct FrontSet {
        DevBuf<float4> scan, scan_ds; DeskewWork dk; VoxelGridWork vg;
        int* d_counts = nullptr; int n_scan_bound = 0, h_n_scan = -1, h_n_ds = -1;   // d_counts: view
    } alt;
    Stream stream_pre;
    Event ev_pre_done, ev_frame_start;
    bool pre_valid = false, frame_start_recorded = false; int pre_index = 0, pre_n = 0; const void* pre_pts = nullptr;
    ~liorf_ctx() {          // no stream may still use what the members release as they are destroyed
        if (!stream) return;                 // nothing was created on the device
        cudaSetDevice(P.device);
        cudaStreamSynchronize(stream);
        if (stream_pre) cudaStreamSynchronize(stream_pre);
        if (stream_map) cudaStreamSynchronize(stream_map);
    }
};

// The two secondary streams are created on first use: a context that only searches the ScanContext database (one lane of a sharded search)
// never needs them, and every stream a process creates competes for the device's hardware channels (CUDA_DEVICE_MAX_CONNECTIONS) — streams
// that share a channel serialise, which turned cross-GPU flag waits of different lanes into a cycle (DESIGN.md §7).
static int make_low_priority_stream(Stream& out) {
    int prio_lo = 0, prio_hi = 0;
    CUDA_TRY(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    if (std::getenv("LIORF_NO_PRIO")) prio_lo = 0;
    CUDA_TRY(stream_create(out, prio_lo));
    return LIORF_OK;
}
static int need_stream_map(liorf_ctx* c) { return c->stream_map ? LIORF_OK : make_low_priority_stream(c->stream_map); }
static int need_stream_pre(liorf_ctx* c) { return c->stream_pre ? LIORF_OK : make_low_priority_stream(c->stream_pre); }

// swaps the current front set with the alternate one (pointer swaps only)
static void front_swap(liorf_ctx* c) {
    std::swap(c->scan, c->alt.scan); std::swap(c->scan_ds, c->alt.scan_ds); std::swap(c->dk, c->alt.dk); std::swap(c->vg, c->alt.vg);
    std::swap(c->d_counts, c->alt.d_counts); std::swap(c->n_scan_bound, c->alt.n_scan_bound);
    std::swap(c->h_n_scan, c->alt.h_n_scan); std::swap(c->h_n_ds, c->alt.h_n_ds);
}
// D2H of the current set's counts together with the shared block: ONE 2 x C_COUNT copy into h_mail[0 : 2 C_COUNT)
static cudaError_t mail_counts(liorf_ctx* c) {
    const int* src = c->d_counts < c->d_shared ? c->d_counts : c->d_shared;
    return cudaMemcpyAsync(c->h_mail.p, src, 2 * C_COUNT * sizeof(int), cudaMemcpyDeviceToHost, c->stream);
}
static void take_counts(liorf_ctx* c) {
    const int so = c->d_counts < c->d_shared ? 0 : C_COUNT, sh = C_COUNT - so;
    c->h_n_scan = c->h_mail.p[so + C_N_SCAN]; c->h_n_ds = c->h_mail.p[so + C_N_DS]; c->h_m_ds = c->h_mail.p[sh + C_M_DS];
}

static void prof_flush(liorf_ctx* c) {           // call only when the stream is idle (after a sync)
    Profiler& p = c->prof;
    int keep = 0;
    for (int i = 0; i < p.pending; ++i) {
        float ms = 0.f;
        if (cudaEventQuery(p.ev[i][1]) == cudaErrorNotReady && keep < PROF_RING / 2) {      // still running on another stream (pipelined front end)
            std::swap(p.ev[i][0], p.ev[keep][0]); std::swap(p.ev[i][1], p.ev[keep][1]); std::swap(p.sec[i], p.sec[keep]); ++keep;
            continue;
        }
        if (cudaEventElapsedTime(&ms, p.ev[i][0], p.ev[i][1]) == cudaSuccess) { p.ms[p.sec[i]] += ms; p.calls[p.sec[i]]++; }
    }
    (void)cudaGetLastError();
    p.pending = keep;
}
struct ProfScope {
    liorf_ctx* c; int slot = -1; cudaStream_t st;
    ProfScope(liorf_ctx* c_, int sec, cudaStream_t st_ = nullptr) : c(c_), st(st_ ? st_ : c_->stream) {
        Profiler& p = c->prof;
        if (!p.enabled || !((p.mask >> sec) & 1u)) return;
        if (!p.created) { for (auto& e : p.ev) { (void)event_create(e[0], cudaEventDefault); (void)event_create(e[1], cudaEventDefault); } p.created = true; }
        if (p.pending == PROF_RING) { cudaStreamSynchronize(c->stream); if (c->stream_map) cudaStreamSynchronize(c->stream_map); prof_flush(c); }
        slot = p.pending++; p.sec[slot] = sec;
        cudaEventRecord(p.ev[slot][0], st);
    }
    ~ProfScope() { if (slot >= 0) cudaEventRecord(c->prof.ev[slot][1], st); }
};

struct Pose6 { float v[6]; };
__global__ void k_set_tf6(float* tf6, Pose6 p) { if (threadIdx.x < 6) tf6[threadIdx.x] = p.v[threadIdx.x]; }
static int upload_pose(liorf_ctx* c, const float* pose6);

static void host_get_transformation(float x, float y, float z, float roll, float pitch, float yaw, float* t) {
    // pcl::getTransformation on the host, exactly where the reference evaluates it (src/mapOptmization.cpp:317)
    float A = std::cos(yaw), B = std::sin(yaw), C = std::cos(pitch), D = std::sin(pitch);
    float E = std::cos(roll), F = std::sin(roll), DE = D * E, DF = D * F;
    t[0] = A * C;  t[1] = A * DF - B * E;  t[2]  = B * F + A * DE;  t[3]  = x;
    t[4] = B * C;  t[5] = A * E + B * DF;  t[6]  = B * DE - A * F;  t[7]  = y;
    t[8] = -D;     t[9] = C * F;           t[10] = C * E;           t[11] = z;
}

// Pinned staging areas are split in two halves used alternately; an event per half tells when its last H2D copy has been
// consumed, so re-use never needs a stream synchronise (the event is normally long complete).
static int stage_slot(liorf_ctx* c, int which) {
    const int turn = c->stage_turn[which] ^= 1;
    if (!c->stage_ev[which][turn]) { if (event_create(c->stage_ev[which][turn], cudaEventDisableTiming) != cudaSuccess) return -1; }
    else if (cudaEventSynchronize(c->stage_ev[which][turn]) != cudaSuccess) return -1;
    return turn;
}
// The local-map chain (extractCloud + VoxelGrid + grid build) runs on stream_map, concurrently with deskew + downsample on
// the main stream.  Every main-stream consumer of the map (solver, hooks, read-backs) joins first.
static int join_map(liorf_ctx* c) {
    if (c->map_pending) { CUDA_TRY(cudaStreamWaitEvent(c->stream, c->ev_map, 0)); c->map_pending = false; }
    return LIORF_OK;
}
static int upload_pose(liorf_ctx* c, const float* pose6) {          // by kernel argument: no pinned staging, no sync
    Pose6 p; std::memcpy(p.v, pose6, sizeof(p.v));
    k_set_tf6<<<1, 32, 0, c->stream>>>(c->d_tf6, p);
    CUDA_TRY(cudaGetLastError());
    return LIORF_OK;
}

static int check_err(liorf_ctx* c) {      // after a stream sync: sticky device-side error flag (bounded look-back spins)
    int e = 0;
    { int rcj = join_map(c); if (rcj) return rcj; }
    CUDA_TRY(cudaMemcpyAsync(c->h_mail.p + 4000, c->d_err, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    prof_flush(c);
    e = c->h_mail.p[4000];
    if (e) {
        fprintf(stderr, "[liorf_b200] device error flag %d (%s)\n", e, e == 5 ? "an mbarrier wait gave up" : e >= 0x30 ? "a peer's exchange flag never arrived: 0x30 + phase, C=0 D=1 KEYS=2" :
                e == 2 ? "solver: a worker / the reducer never arrived" : "look-back predecessor never arrived");
        return LIORF_ERR_DEVICE_FLAG;
    }
    return LIORF_OK;
}

static int read_counts(liorf_ctx* c) {
    { int rcj = join_map(c); if (rcj) return rcj; }
    CUDA_TRY(mail_counts(c));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    prof_flush(c);
    take_counts(c);
    return LIORF_OK;
}

static int sc_reserve(liorf_ctx* c, int n) {
    int rc;
    ScDatabase& db = *c->sc_db;
    if (c->sc_borrowed()) return (size_t)n * SC_RING <= db.keys.cap ? LIORF_OK : LIORF_ERR_STATE;      // a borrowed database is read-only here
    if ((rc = db.desc.reserve((size_t)n * SC_DESC, c->stream, true)) || (rc = db.sk.reserve((size_t)n * SC_SECTOR, c->stream, true)) ||
        (rc = db.cn.reserve((size_t)n * SC_SECTOR, c->stream, true)) || (rc = db.keys.reserve((size_t)n * SC_RING, c->stream, true))) return rc;
    return LIORF_OK;
}


extern "C" {

const char* liorf_version(void) { return "liorf_b200 0.1 (sm_100a)"; }

void liorf_default_params(liorf_params* p) {      // config/kitti.yaml
    if (!p) return;
    std::memset(p, 0, sizeof(*p));
    p->N_SCAN = 64; p->downsampleRate = 2; p->point_filter_num = 5;
    p->lidarMinRange = 1.0f; p->lidarMaxRange = 1000.0f;
    p->mappingSurfLeafSize = 0.4f; p->surroundingKeyframeMapLeafSize = 0.5f; p->surroundingKeyframeSearchRadius = 50.0f;
    p->grid_dim_x = 256; p->grid_dim_y = 256; p->grid_dim_z = 32; p->device = 0;
}

static bool is_pow2(int v) { return v > 0 && (v & (v - 1)) == 0; }

int liorf_create(const liorf_params* p, liorf_ctx** out) {
    LIORF_NVTX;
    if (!p || !out) return LIORF_ERR_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        fprintf(stderr, "[liorf_b200] no CUDA device: this library has no CPU path\n");
        return LIORF_ERR_CUDA;
    }
    std::unique_ptr<liorf_ctx> c(new (std::nothrow) liorf_ctx());      // every early return below frees what was created so far
    if (!c) return LIORF_ERR_ARG;
    c->P = *p;
    c->host_timing = std::getenv("LIORF_HOST_TIMING") != nullptr;
    c->use_graphs = std::getenv("LIORF_NO_GRAPH") == nullptr;
    if (c->P.grid_dim_x == 0) c->P.grid_dim_x = 256;
    if (c->P.grid_dim_y == 0) c->P.grid_dim_y = 256;
    if (c->P.grid_dim_z == 0) c->P.grid_dim_z = 32;
    if (!is_pow2(c->P.grid_dim_x) || !is_pow2(c->P.grid_dim_y) || !is_pow2(c->P.grid_dim_z) || c->P.grid_dim_x < 4) return LIORF_ERR_ARG;
    if (c->P.downsampleRate < 1 || c->P.point_filter_num < 1) return LIORF_ERR_ARG;
    c->grid.dims = GridDims{c->P.grid_dim_x, c->P.grid_dim_y, c->P.grid_dim_z};
    CUDA_TRY(cudaSetDevice(c->P.device));
    cudaDeviceProp prop; CUDA_TRY(cudaGetDeviceProperties(&prop, c->P.device));
    c->num_sms = prop.multiProcessorCount;
    // The reducer CTA of the solver collects the partial sums of at most S2M_MAX_WORKERS workers (a register array sized at compile
    // time); a grid of num_sms CTAs has num_sms - 1 workers.  A B200 (148 SMs) is within the limit, so this refusal never runs there.
    if (c->num_sms - 1 > S2M_MAX_WORKERS) {
        fprintf(stderr, "[liorf_b200] %d SMs: the solver supports at most %d (raise S2M_MAX_WORKERS in scan2map.cuh)\n", c->num_sms, S2M_MAX_WORKERS + 1);
        return LIORF_ERR_CUDA;
    }
    // the main stream carries the latency-critical chain (deskew → downsample → solver); giving it the highest priority lets
    // its large-footprint CTAs (single-CTA VoxelGrid, one-CTA-per-SM solver) claim SMs from the concurrent local-map chain
    int prio_lo = 0, prio_hi = 0;
    CUDA_TRY(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    if (std::getenv("LIORF_NO_PRIO")) prio_lo = prio_hi = 0;
    CUDA_TRY(stream_create(c->stream, prio_hi));
    CUDA_TRY(dev_alloc(c->d_counts_base, 3 * C_COUNT));
    CUDA_TRY(cudaMemset(c->d_counts_base, 0, 3 * C_COUNT * sizeof(int)));
    c->d_counts = c->d_counts_base; c->d_shared = c->d_counts_base + C_COUNT; c->alt.d_counts = c->d_counts_base + 2 * C_COUNT;
    CUDA_TRY(dev_alloc(c->d_misc, 64));
    CUDA_TRY(cudaMemset(c->d_misc, 0, 64 * sizeof(int)));
    c->d_err = c->d_misc + 0;
    {
        unsigned long long init[16]; for (auto& v : init) v = TICKET_INIT;
        CUDA_TRY(dev_alloc(c->d_tick, 16));
        CUDA_TRY(cudaMemcpy(c->d_tick, init, sizeof(init), cudaMemcpyHostToDevice));
    }
    c->vg.mm_counter = c->d_misc + 1;
    c->vg.sort.ticket = c->d_tick + 0; c->vg.sort.err_flag = c->d_err;
    c->vg.scan.ticket = c->d_tick + 1; c->vg.scan.err_flag = c->d_err;
    c->grid.scan.ticket = c->d_tick + 2; c->grid.scan.err_flag = c->d_err;
    c->dk.scan.ticket = c->d_tick + 3; c->dk.scan.err_flag = c->d_err;
    c->combine_scan.ticket = c->d_tick + 4; c->combine_scan.err_flag = c->d_err;
    CUDA_TRY(dev_alloc(c->vg.meta, 1));
    for (VoxelGridWork* vw : {&c->vg, &c->vg_map, &c->alt.vg}) {          // grid-barrier words of the one-kernel VoxelGrid
        CUDA_TRY(dev_alloc(vw->fused_bar, 2)); CUDA_TRY(cudaMemset(vw->fused_bar, 0, 2 * sizeof(unsigned))); vw->err_flag = c->d_err;
    }
    CUDA_TRY(event_create(c->ev_main, cudaEventDisableTiming));
    CUDA_TRY(event_create(c->ev_map, cudaEventDisableTiming));
    CUDA_TRY(dev_alloc(c->vg_map.meta, 1));
    c->vg_map.mm_counter = c->d_misc + 10;
    c->vg_map.sort.ticket = c->d_tick + 5; c->vg_map.sort.err_flag = c->d_err;
    c->vg_map.scan.ticket = c->d_tick + 6; c->vg_map.scan.err_flag = c->d_err;
    c->icp_grid.scan.ticket = c->d_tick + 7; c->icp_grid.scan.err_flag = c->d_err;
    c->icpb.sort.ticket = c->d_tick + 11; c->icpb.sort.err_flag = c->d_err;
    c->icpb.scan.ticket = c->d_tick + 12; c->icpb.scan.err_flag = c->d_err;
    c->icpb.grid_scan.ticket = c->d_tick + 13; c->icpb.grid_scan.err_flag = c->d_err;
    CUDA_TRY(dev_alloc(c->icpb.d_flags, 2));
    CUDA_TRY(dev_alloc(c->dk.start_inv, 12));
    c->dk.first_kept = c->d_counts + C_FIRST_KEPT;
    // the alternate front set: its own look-back tickets, VoxelGrid meta and deskew scalars
    c->alt.vg.mm_counter = c->d_misc + 20;
    c->alt.vg.sort.ticket = c->d_tick + 8; c->alt.vg.sort.err_flag = c->d_err;
    c->alt.vg.scan.ticket = c->d_tick + 9; c->alt.vg.scan.err_flag = c->d_err;
    c->alt.dk.scan.ticket = c->d_tick + 10; c->alt.dk.scan.err_flag = c->d_err;
    CUDA_TRY(dev_alloc(c->alt.vg.meta, 1));
    CUDA_TRY(dev_alloc(c->alt.dk.start_inv, 12));
    c->alt.dk.first_kept = c->alt.d_counts + C_FIRST_KEPT;
    CUDA_TRY(event_create(c->ev_pre_done, cudaEventDisableTiming));
    CUDA_TRY(event_create(c->ev_frame_start, cudaEventDisableTiming));
    { int rc = c->h_mail.reserve((65536 + 2 * 65536) / sizeof(int)); if (rc) return rc; }
    CUDA_TRY(dev_alloc(c->d_tf6, 6));
    CUDA_TRY(cudaMemset(c->d_tf6, 0, 6 * sizeof(float)));
    CUDA_TRY(dev_alloc(c->d_lm, 1));
    CUDA_TRY(cudaMemset(c->d_lm, 0, sizeof(LMDeviceState)));
    CUDA_TRY(dev_alloc(c->d_trace, 1));
    CUDA_TRY(cudaMemset(c->d_trace, 0, sizeof(S2MTrace)));
    CUDA_TRY(dev_alloc(c->d_lm_out, 48));
    int occ = 0;
    CUDA_TRY(cudaFuncSetAttribute(k_scan2map_persistent, cudaFuncAttributeMaxDynamicSharedMemorySize, S2MP_SMEM));
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_scan2map_persistent, S2MP_BLOCK, S2MP_SMEM));
    if (occ < 1) { fprintf(stderr, "[liorf_b200] persistent kernel does not fit\n"); return LIORF_ERR_CUDA; }
    // liorf_process_frame runs the solver on one persistent CTA per SM of all but S2M_SPARE_SMS SMs.  The solver's CTA owns its SM
    // outright (512 threads x 128 registers = the whole register file), so the SMs it leaves free are where the NEXT frame's
    // cloudHandler + downsample (stream_pre) run while it iterates.  The solve is latency-bound (one round of <= 128 queries per CTA up
    // to ~17k points), so the narrower grid costs nothing at the KITTI sizes.  The grid is the same with and without look-ahead, so
    // those two give bit-identical results.  The per-function calls (liorf_scan2map_optimization[_async]) launch num_sms CTAs instead:
    // the grid width decides which worker serves each query, how the fp64 partial sums are grouped and from which scan size on the
    // per-query state moves to global memory, so their results may differ from liorf_process_frame's in the last bits.
    // liorf_debug_s2m_grid sets the width of both for tests.
    {
        int spare = S2M_SPARE_SMS;
        if (const char* e = std::getenv("LIORF_SOLVER_SPARE_SMS")) spare = std::atoi(e);
        if (spare < 0) spare = 0;
        c->s2m_grid = c->num_sms - spare; if (c->s2m_grid < 2) c->s2m_grid = c->num_sms;      // >= 2: workers + the reducer CTA
        // the local-map VoxelGrid stays on the multi-kernel path: at 300-650 k points the one-kernel version is no faster (its multi-tile chunks
        // sweep the keys twice per pass: 0.142-0.228 ms against 0.144-0.154 ms for the KITTI map, 0.466 against 0.288 ms for the 2.3 M-point OS1-128
        // selection, sequence 0.198 against 0.204 ms/frame) and two cooperative grids would compete for the SMs;
        // LIORF_MAP_VG_GRID = CTAs of the one-kernel path for experiments
        c->map_vg_grid = 0;
        if (const char* e = std::getenv("LIORF_MAP_VG_GRID")) c->map_vg_grid = std::atoi(e);
        if (c->map_vg_grid > c->num_sms) c->map_vg_grid = c->num_sms;
    }
    CUDA_TRY(dev_alloc(c->d_partial, (size_t)2 * c->num_sms * NPROD));
    CUDA_TRY(dev_alloc(c->d_mail, 1));
    // hand-off words of the solver (epoch-tagged: zero never matches an epoch, launch sequence numbers start at 1)
    CUDA_TRY(dev_alloc(c->d_wpart, (size_t)c->num_sms * NPROD));
    CUDA_TRY(cudaMemset(c->d_wpart, 0, (size_t)c->num_sms * NPROD * sizeof(ulonglong2)));
    CUDA_TRY(dev_alloc(c->d_res, 8));
    CUDA_TRY(cudaMemset(c->d_res, 0, 8 * sizeof(unsigned long long)));
    CUDA_TRY(dev_alloc(c->d_bins, SC_DESC));
    {   // arm the ScanContext bins with the NO_POINT code
        std::vector<unsigned> init(SC_DESC);
        float f = -1000.f; unsigned u; std::memcpy(&u, &f, 4); u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
        for (auto& v : init) v = u;
        CUDA_TRY(cudaMemcpy(c->d_bins, init.data(), SC_DESC * sizeof(unsigned), cudaMemcpyHostToDevice));
    }
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    *out = c.release();
    return LIORF_OK;
}

void liorf_destroy(liorf_ctx* c) {
    if (!c) return;
    if (c->host_timing && c->host_frames > 0) {
        const char* nm[6] = {"enqueue deskew", "select+enqueue map", "enqueue downsample", "enqueue solver", "wait pose (sync)", "keyframe+sc+loop"};
        fprintf(stderr, "[liorf_b200] host timeline per frame over %lld frames:", c->host_frames);
        for (int k = 0; k < 6; ++k) fprintf(stderr, "  %s %.1f us;", nm[k], c->host_us[k] / c->host_frames);
        fprintf(stderr, "\n[liorf_b200] keyframe tail per frame: save+add keyframe %.1f; extract_nearby(next) %.1f; enqueue next map %.1f; ScanContext make %.1f; loop detection %.1f us",
                c->host_us[6] / c->host_frames, c->host_us[7] / c->host_frames, c->host_us[8] / c->host_frames, c->host_us[9] / c->host_frames, c->host_us[10] / c->host_frames);
        fprintf(stderr, "\n[liorf_b200] GPU timeline (us after frame start): deskew done %.1f; map+grid done %.1f; downsample done %.1f; joined %.1f; solver done %.1f\n",
                1e3 * c->tl_ms[1] / c->host_frames, 1e3 * c->tl_ms[2] / c->host_frames, 1e3 * c->tl_ms[3] / c->host_frames, 1e3 * c->tl_ms[4] / c->host_frames,
                1e3 * c->tl_ms[5] / c->host_frames);
    }
    delete c;
}

int liorf_sync(liorf_ctx* c) { if (!c) return LIORF_ERR_ARG; CUDA_TRY(cudaSetDevice(c->P.device)); return check_err(c); }
void* liorf_stream(liorf_ctx* c) { return c ? (void*)c->stream : nullptr; }

// ------------------------------------------------------------------------------------------------ imageProjection
static int project_common(liorf_ctx* c, const RawPoint* d_raw, int n, double t0, const double* imu_time, const double* rx, const double* ry,
                          const double* rz, int imu_ptr, int deskew_enabled, int* d_kept_index) {
    int rc;
    // `i % point_filter_num == 0` is necessary for a point to survive (:591) ⇒ a host-side bound on the kept count
    const int kept_bound = n > 0 ? (n + c->P.point_filter_num - 1) / c->P.point_filter_num : 0;
    if ((rc = c->scan.reserve(kept_bound > 0 ? kept_bound : 1))) return rc;
    if ((rc = c->dk.kept.reserve(kept_bound > 0 ? kept_bound : 1))) return rc;
    c->n_scan_bound = kept_bound; c->h_n_scan = -1; c->h_n_ds = -1;
    if (n <= 0) { CUDA_TRY(cudaMemsetAsync(c->d_counts + C_N_SCAN, 0, sizeof(int), c->stream)); c->h_n_scan = 0; return LIORF_OK; }
    ImuTable T{nullptr, nullptr, nullptr, nullptr, 0};
    if (deskew_enabled) {
        if (imu_ptr < 0 || !imu_time || !rx || !ry || !rz) return LIORF_ERR_ARG;
        const int rows = imu_ptr + 1;
        if ((rc = c->dk.imu.reserve((size_t)4 * rows))) return rc;
        if ((size_t)4 * rows * sizeof(double) > 65536) return LIORF_ERR_ARG;        // queueLength = 2000 rows (src/imageProjection.cpp:62) = 64000 B
        const int slot = stage_slot(c, 1); if (slot < 0) return LIORF_ERR_CUDA;
        double* stage = reinterpret_cast<double*>(c->h_mail.p + 16384 + slot * 16384);   // pinned staging (two 64 KB halves above the mailbox)
        std::memcpy(stage, imu_time, rows * sizeof(double)); std::memcpy(stage + rows, rx, rows * sizeof(double));
        std::memcpy(stage + 2 * rows, ry, rows * sizeof(double)); std::memcpy(stage + 3 * rows, rz, rows * sizeof(double));
        CUDA_TRY(cudaMemcpyAsync(c->dk.imu.p, stage, (size_t)4 * rows * sizeof(double), cudaMemcpyHostToDevice, c->stream));
        CUDA_TRY(cudaEventRecord(c->stage_ev[1][slot], c->stream));
        T = ImuTable{c->dk.imu.p, c->dk.imu.p + rows, c->dk.imu.p + 2 * rows, c->dk.imu.p + 3 * rows, imu_ptr};
    }
    DeskewParams DP{c->P.lidarMinRange, c->P.lidarMaxRange, c->P.N_SCAN, c->P.downsampleRate, c->P.point_filter_num};
    ProfScope ps(c, SEC_DESKEW); c->launches += 3;
    k_first_kept<<<1, 1024, 0, c->stream>>>(d_raw, n, DP, t0, T, deskew_enabled, c->dk.start_inv, c->dk.first_kept);
    int* kept = d_kept_index ? d_kept_index : c->dk.kept.p;
    rc = launch_scan(Count::of_host(n), DeskewLoad{d_raw, DP}, DeskewStore{kept}, c->dk.scan, (unsigned*)(c->d_counts + C_N_SCAN), c->stream);
    if (rc) return rc;
    k_deskew_points<<<(kept_bound + 127) / 128, 128, 0, c->stream>>>(d_raw, kept, c->d_counts + C_N_SCAN, t0, T, deskew_enabled, c->dk.start_inv, c->scan.p);
    CUDA_TRY(cudaGetLastError());
    return LIORF_OK;
}

int liorf_project_point_cloud(liorf_ctx* c, const liorf_point_xyzirt* pts, int n, double t0, const double* imu_time, const double* rx,
                              const double* ry, const double* rz, int imu_ptr, int deskew_enabled, liorf_point* out, int* n_out, int* kept_index) {
    LIORF_NVTX;
    if (!c || n < 0 || (n > 0 && !pts)) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    int rc;
    if ((rc = c->dk.raw.reserve(n > 0 ? n : 1))) return rc;
    if (n > 0) CUDA_TRY(cudaMemcpyAsync(c->dk.raw.p, pts, (size_t)n * sizeof(RawPoint), cudaMemcpyHostToDevice, c->stream));
    int* d_ki = nullptr;
    if (kept_index) { if ((rc = c->membership.reserve(n > 0 ? n : 1))) return rc; d_ki = c->membership.p; }
    if ((rc = project_common(c, c->dk.raw.p, n, t0, imu_time, rx, ry, rz, imu_ptr, deskew_enabled, d_ki))) return rc;
    if (!out && !n_out && !kept_index) return LIORF_OK;          // stay asynchronous: the cloud feeds downsampleCurrentScan on the device
    if ((rc = read_counts(c))) return rc;
    if (n_out) *n_out = c->h_n_scan;
    if (out && c->h_n_scan > 0) CUDA_TRY(cudaMemcpyAsync(out, c->scan.p, (size_t)c->h_n_scan * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
    if (kept_index && c->h_n_scan > 0) CUDA_TRY(cudaMemcpyAsync(kept_index, d_ki, (size_t)c->h_n_scan * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    return check_err(c);
}

int liorf_project_point_cloud_dev(liorf_ctx* c, const void* d_pts, int n, double t0, const double* imu_time, const double* rx, const double* ry,
                                  const double* rz, int imu_ptr, int deskew_enabled) {
    LIORF_NVTX;
    if (!c || n < 0 || (n > 0 && !d_pts)) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    return project_common(c, (const RawPoint*)d_pts, n, t0, imu_time, rx, ry, rz, imu_ptr, deskew_enabled, nullptr);
}

// ------------------------------------------------------------------------------------------------ mapOptimization
static Count map_count(liorf_ctx* c);
static int set_scan_common(liorf_ctx* c, const void* src, int n, cudaMemcpyKind kind) {
    int rc;
    if ((rc = c->scan.reserve(n > 0 ? n : 1))) return rc;
    if (n > 0) CUDA_TRY(cudaMemcpyAsync(c->scan.p, src, (size_t)n * sizeof(float4), kind, c->stream));
    c->h_mail.p[100] = n;
    // count goes through a kernel-visible device int
    CUDA_TRY(cudaMemcpyAsync(c->d_counts + C_N_SCAN, &c->h_mail.p[100], sizeof(int), cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    c->n_scan_bound = n; c->h_n_scan = n; c->h_n_ds = -1;
    return LIORF_OK;
}
// cloud_info.cloud_deskewed as mapOptimization receives it (msg/cloud_info.msg:27; pcl::fromROSMsg into PointXYZI, include/utility.h:61):
// a sensor_msgs/PointCloud2 data block with `point_step` bytes per point (32 for PCL's padded PointXYZI), x, y, z as three consecutive floats
// at offset_xyz and the intensity float at offset_intensity (16).  The block is copied as it is and unpacked to the library's 16-byte points
// on the device, so a ROS shim can hand msg.data straight to the library.
__global__ void __launch_bounds__(256) k_unpack_strided(const unsigned char* __restrict__ raw, int n, int step, int off_xyz, int off_i, float4* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned char* p = raw + (size_t)i * step;
    float4 o;
    if (((step | off_xyz | off_i) & 3) == 0 && (reinterpret_cast<size_t>(raw) & 3) == 0) {
        const float* f = reinterpret_cast<const float*>(p + off_xyz);
        o.x = f[0]; o.y = f[1]; o.z = f[2]; o.w = *reinterpret_cast<const float*>(p + off_i);
    } else {                                                       // unaligned layouts: byte-wise
        float v[4];
        for (int k = 0; k < 3; ++k) { unsigned u = 0; for (int b = 0; b < 4; ++b) u |= (unsigned)p[off_xyz + 4 * k + b] << (8 * b); v[k] = __uint_as_float(u); }
        { unsigned u = 0; for (int b = 0; b < 4; ++b) u |= (unsigned)p[off_i + b] << (8 * b); v[3] = __uint_as_float(u); }
        o = make_float4(v[0], v[1], v[2], v[3]);
    }
    out[i] = o;
}
int liorf_set_current_scan_strided(liorf_ctx* c, const void* data, int n, int point_step, int offset_xyz, int offset_intensity, int data_on_device) {
    LIORF_NVTX;
    if (!c || n < 0 || (n > 0 && !data) || point_step < 16 || offset_xyz < 0 || offset_intensity < 0 || offset_xyz + 12 > point_step || offset_intensity + 4 > point_step)
        return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    int rc;
    if ((rc = c->scan.reserve(n > 0 ? n : 1))) return rc;
    const unsigned char* d_raw = (const unsigned char*)data;
    if (!data_on_device && n > 0) {
        const size_t bytes = (size_t)n * point_step;
        if ((rc = c->dk.raw.reserve((bytes + sizeof(RawPoint) - 1) / sizeof(RawPoint)))) return rc;       // the raw-scan staging buffer doubles as the byte staging area
        CUDA_TRY(cudaMemcpyAsync(c->dk.raw.p, data, bytes, cudaMemcpyHostToDevice, c->stream));
        d_raw = reinterpret_cast<const unsigned char*>(c->dk.raw.p);
    }
    if (n > 0) k_unpack_strided<<<(n + 255) / 256, 256, 0, c->stream>>>(d_raw, n, point_step, offset_xyz, offset_intensity, c->scan.p);
    CUDA_TRY(cudaGetLastError());
    c->h_mail.p[100] = n;
    CUDA_TRY(cudaMemcpyAsync(c->d_counts + C_N_SCAN, &c->h_mail.p[100], sizeof(int), cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    c->n_scan_bound = n; c->h_n_scan = n; c->h_n_ds = -1; c->launches += 1;
    return LIORF_OK;
}
int liorf_set_current_scan(liorf_ctx* c, const liorf_point* scan, int n) {
    LIORF_NVTX;
    if (!c || n < 0 || (n > 0 && !scan)) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    return set_scan_common(c, scan, n, cudaMemcpyHostToDevice);
}
int liorf_set_current_scan_dev(liorf_ctx* c, const void* d_scan, int n) {
    LIORF_NVTX;
    if (!c || n < 0 || (n > 0 && !d_scan)) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    return set_scan_common(c, d_scan, n, cudaMemcpyDeviceToDevice);
}

// coop_grid: CTAs of the one-kernel VoxelGrid (all SMs for a standalone call, the SMs the solver leaves free for the look-ahead front end)
static int downsample_async(liorf_ctx* c, int* d_membership, int coop_grid) {
    int rc;
    const int nb = c->n_scan_bound;
    if ((rc = c->scan_ds.reserve(nb > 0 ? nb : 1))) return rc;
    c->h_n_ds = -1;
    Count cnt = c->h_n_scan >= 0 ? Count::of_host(c->h_n_scan) : Count::of_dev(c->d_counts + C_N_SCAN, nb);
    ProfScope ps(c, SEC_DOWNSAMPLE);
    rc = voxel_grid_device(c->scan.p, cnt, c->P.mappingSurfLeafSize, c->scan_ds.p, c->d_counts + C_N_DS, d_membership, nullptr, c->vg, c->stream, coop_grid);
    c->launches += c->vg.last_launches;
    return rc;
}

int liorf_downsample_current_scan(liorf_ctx* c, liorf_point* out, int* n_ds, int* membership) {
    LIORF_NVTX;
    if (!c) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    int rc;
    int* d_mem = nullptr;
    if (membership) { if ((rc = c->membership.reserve(c->n_scan_bound > 0 ? c->n_scan_bound : 1))) return rc; d_mem = c->membership.p; }
    if ((rc = downsample_async(c, d_mem, c->num_sms))) return rc;
    if (!out && !n_ds && !membership) return LIORF_OK;           // stay asynchronous
    if ((rc = read_counts(c))) return rc;
    if (n_ds) *n_ds = c->h_n_ds;
    if (out && c->h_n_ds > 0) CUDA_TRY(cudaMemcpyAsync(out, c->scan_ds.p, (size_t)c->h_n_ds * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
    if (membership && c->h_n_scan > 0) CUDA_TRY(cudaMemcpyAsync(membership, d_mem, (size_t)c->h_n_scan * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    return check_err(c);
}

int liorf_voxel_grid(liorf_ctx* c, const liorf_point* in, int n, float leaf, liorf_point* out, int* n_out, int* membership, int* out_keys) {
    LIORF_NVTX;
    if (!c || n < 0 || (n > 0 && !in) || !n_out) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    int rc;
    if ((rc = join_map(c))) return rc;
    const int cap = n > 0 ? n : 1;
    if ((rc = c->map_raw.reserve(cap))) return rc;       // scratch in / out (does not disturb the scan or the map)
    DevBuf<float4> tmp_out; if ((rc = tmp_out.reserve(cap))) return rc;
    if ((rc = c->membership.reserve(cap))) return rc;
    if ((rc = c->out_keys.reserve(cap))) return rc;
    if (n > 0) CUDA_TRY(cudaMemcpyAsync(c->map_raw.p, in, (size_t)n * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
    rc = voxel_grid_device(c->map_raw.p, Count::of_host(n), leaf, tmp_out.p, c->d_counts + C_NSEL, c->membership.p, c->out_keys.p, c->vg, c->stream, c->vg_ctas ? c->vg_ctas : c->num_sms);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->h_mail.p + 200, c->d_counts + C_NSEL, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    int no = c->h_mail.p[200]; *n_out = no;
    if (out && no > 0) CUDA_TRY(cudaMemcpyAsync(out, tmp_out.p, (size_t)no * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
    if (membership && n > 0) CUDA_TRY(cudaMemcpyAsync(membership, c->membership.p, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    if (out_keys && no > 0) CUDA_TRY(cudaMemcpyAsync(out_keys, c->out_keys.p, (size_t)no * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    rc = check_err(c);
    c->map_valid = false;                                 // map_raw scratch was reused
    return rc;
}

static int append_keyframe(liorf_ctx* c, const float4* d_src, const float4* h_src, int n, const float pose6[6], double time) {
    int rc;
    if ((rc = c->kf_points.reserve(c->kf_used + (size_t)(n > 0 ? n : 1), c->stream, true))) return rc;
    if (n > 0) {
        if (d_src) CUDA_TRY(cudaMemcpyAsync(c->kf_points.p + c->kf_used, d_src, (size_t)n * sizeof(float4), cudaMemcpyDeviceToDevice, c->stream));
        else CUDA_TRY(cudaMemcpyAsync(c->kf_points.p + c->kf_used, h_src, (size_t)n * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
    }
    Keyframe k; k.off = c->kf_used; k.count = n; std::memcpy(k.pose, pose6, sizeof(k.pose)); k.time = time;
    c->kfs.push_back(k); c->kf_used += (size_t)n;
    ++c->pose_version;
    return (int)c->kfs.size() - 1;
}
int liorf_add_keyframe(liorf_ctx* c, const float pose6[6], double time) {
    LIORF_NVTX;
    if (!c || !pose6) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    int rc;
    if (c->h_n_ds < 0 && (rc = read_counts(c))) return rc;
    return append_keyframe(c, c->scan_ds.p, nullptr, c->h_n_ds, pose6, time);
}
int liorf_add_keyframe_cloud(liorf_ctx* c, const liorf_point* cloud, int n, const float pose6[6], double time) {
    LIORF_NVTX;
    if (!c || !pose6 || n < 0 || (n > 0 && !cloud)) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    int id = append_keyframe(c, nullptr, (const float4*)cloud, n, pose6, time);
    if (id >= 0) CUDA_TRY(cudaStreamSynchronize(c->stream));      // host buffer may be reused by the caller
    return id;
}
int liorf_update_keyframe_pose(liorf_ctx* c, int id, const float pose6[6]) {
    LIORF_NVTX;
    if (!c || id < 0 || id >= (int)c->kfs.size() || !pose6) return LIORF_ERR_ARG;
    std::memcpy(c->kfs[id].pose, pose6, 6 * sizeof(float)); ++c->pose_version;
    return LIORF_OK;
}
int liorf_num_keyframes(liorf_ctx* c) { return c ? (int)c->kfs.size() : LIORF_ERR_ARG; }

int liorf_extract_surrounding_keyframes(liorf_ctx* c, const int* ids, int n_ids, int* m_ds) {
    LIORF_NVTX;
    if (!c || n_ids < 0 || (n_ids > 0 && !ids)) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    if (c->kfs.empty()) return LIORF_ERR_STATE;                  // extractSurroundingKeyFrames returns early (:1048)
    int rc;
    std::vector<int> sel; sel.reserve(n_ids);                    // ids verbatim: the :1018 distance gate lives in liorf_extract_nearby, which knows the
    for (int i = 0; i < n_ids; ++i) {                            // positions extractCloud tests (voxel centroids for the thinned radius set)
        if (ids[i] < 0 || ids[i] >= (int)c->kfs.size()) return LIORF_ERR_ARG;
        sel.push_back(ids[i]);
    }
    // the map is a pure function of (selection, poses): identical request ⇒ keep the resident map and grid
    if (c->map_valid && sel == c->last_sel && c->last_sel_version == c->pose_version) {
        if (m_ds) { if (c->h_m_ds < 0 && (rc = read_counts(c))) return rc; *m_ds = c->h_m_ds; }
        return LIORF_OK;
    }
    const int ns = (int)sel.size();
    if ((size_t)ns + 1 > c->h_sel.cap / 2) {
        CUDA_TRY(cudaStreamSynchronize(c->stream));
        if (c->stream_map) CUDA_TRY(cudaStreamSynchronize(c->stream_map));
        if ((rc = c->h_sel.reserve((size_t)2 * (2 * ns + 64)))) return rc;
    }
    if ((rc = c->d_sel.reserve(ns + 1))) return rc;
    const int slot = stage_slot(c, 0); if (slot < 0) return LIORF_ERR_CUDA;
    KfSel* hsel = c->h_sel.p + (size_t)slot * (c->h_sel.cap / 2);      // entry 0 = header {nsel, total}, selections from entry 1
    long long total = 0;
    for (int i = 0; i < ns; ++i) {
        const Keyframe& k = c->kfs[sel[i]];
        KfSel& s = hsel[1 + i];
        s.src_off = (int)k.off; s.count = k.count; s.dst_off = (int)total; s.pad = 0;
        host_get_transformation(k.pose[3], k.pose[4], k.pose[5], k.pose[0], k.pose[1], k.pose[2], s.t);
        total += k.count;
    }
    if (total > 0x7fffffffLL) return LIORF_ERR_ARG;
    const int tot = (int)total;
    std::memset(&hsel[0], 0, sizeof(KfSel)); hsel[0].src_off = ns; hsel[0].count = tot;
    // graph path: grids are sized from the bucket bound, the exact total is read from the header on the device
    const bool graphs = c->use_graphs && tot > VGS_CAP;
    const int bucket = graphs ? (tot + 65535) / 65536 : 0;
    const int bound = graphs ? bucket * 65536 : tot;
    if ((rc = c->map_raw.reserve(bound > 0 ? bound : 1))) return rc;
    if ((rc = c->map_ds.reserve(bound > 0 ? bound : 1))) return rc;
    // fork: everything enqueued so far on the main stream (keyframe copies, the previous solve that still reads the old map)
    // happens-before the map chain
    if ((rc = need_stream_map(c))) return rc;
    cudaStream_t ms = c->stream_map;
    CUDA_TRY(cudaEventRecord(c->ev_main, c->stream));
    CUDA_TRY(cudaStreamWaitEvent(ms, c->ev_main, 0));
    CUDA_TRY(cudaMemcpyAsync(c->d_sel.p, hsel, (size_t)(ns + 1) * sizeof(KfSel), cudaMemcpyHostToDevice, ms));
    CUDA_TRY(cudaEventRecord(c->stage_ev[0][slot], ms));
    const Count cnt_raw = graphs ? Count::of_dev(&c->d_sel.p[0].count, bound) : Count::of_host(tot);
    auto enqueue_vg = [&]() -> int {
        if (tot > 0) {
            if (graphs) k_transform_concat_hdr<<<(bound + 255) / 256, 256, 0, ms>>>(c->kf_points.p, c->d_sel.p, c->map_raw.p);
            else k_transform_concat<<<(tot + 255) / 256, 256, 0, ms>>>(c->kf_points.p, c->d_sel.p + 1, ns, tot, c->map_raw.p);
        }
        return voxel_grid_device(c->map_raw.p, cnt_raw, c->P.surroundingKeyframeMapLeafSize, c->map_ds.p, c->d_shared + C_M_DS, nullptr, nullptr, c->vg_map, ms, c->map_vg_grid);
    };
    auto enqueue_grid = [&]() -> int { return build_map_grid(c->map_ds.p, Count::of_dev(c->d_shared + C_M_DS, bound), c->grid, ms); };
    if (!graphs) {
        { ProfScope ps(c, SEC_MAP_BUILD, ms); c->launches += 10; if ((rc = enqueue_vg())) return rc; }
        { ProfScope ps(c, SEC_GRID_BUILD, ms); c->launches += 3; if ((rc = enqueue_grid())) return rc; }
    } else {
        liorf_ctx::MapGraphs& G = c->map_graphs[bucket];
        // every buffer the chain touches, sized for the bucket BEFORE capture (no allocation or memset may happen inside it)
        VoxelGridWork& w = c->vg_map; MapGrid& gr = c->grid;
        const int nc = grid_cells(gr.dims);
        int mmb = (bound + VG_MM_BLOCK * 8 - 1) / (VG_MM_BLOCK * 8); if (mmb > kNumSMs) mmb = kNumSMs;
        if ((rc = w.pts_sorted.reserve(bound)) || (rc = w.cta_hist.reserve((size_t)kNumSMs * RADIX)) || (rc = w.cta_heads.reserve(kNumSMs)) || (rc = w.partial.reserve((size_t)kNumSMs * 6))) return rc;
        if ((rc = w.partial.reserve((size_t)mmb * 6)) || (rc = w.keys.reserve(bound)) || (rc = w.seg_start.reserve((size_t)bound + 1)) ||
            (rc = w.sort.keys_alt.reserve(bound)) || (rc = w.sort.vals_a.reserve(bound)) || (rc = w.sort.vals_b.reserve(bound)) || (rc = w.sort.hist.reserve(4 * RADIX)) ||
            (rc = reserve_zeroed(w.sort.status, (size_t)((bound + SORT_TILE - 1) / SORT_TILE) * RADIX, ms)) ||
            (rc = reserve_zeroed(w.scan.status, (size_t)(bound + SCAN_TILE - 1) / SCAN_TILE, ms)) ||
            (rc = gr.counts.reserve(nc)) || (rc = gr.cell_start.reserve((size_t)nc + 1)) || (rc = gr.sorted.reserve(bound)) ||
            (rc = reserve_zeroed(gr.scan.status, (size_t)(nc + 512 * 16 - 1) / (512 * 16), ms))) return rc;
        if (!gr.counts_clean) { CUDA_TRY(cudaMemsetAsync(gr.counts.p, 0, (size_t)nc * sizeof(unsigned), ms)); gr.counts_clean = true; }
        const void* sig[20] = {c->kf_points.p, c->d_sel.p, c->map_raw.p, c->map_ds.p, w.partial.p, w.keys.p, w.seg_start.p, w.sort.keys_alt.p, w.sort.vals_a.p,
                               w.sort.vals_b.p, w.sort.hist.p, w.sort.status.p, w.scan.status.p, gr.counts.p, gr.cell_start.p, gr.sorted.p, gr.scan.status.p,
                               w.meta, (const void*)(size_t)(w.force_large | (w.force_multi << 1) | (c->map_vg_grid << 2)), w.pts_sorted.p};
        if (G.vg && std::memcmp(sig, G.sig, sizeof(sig)) != 0) { G.vg.reset(); G.grid.reset(); }
        if (!G.vg) {
            const bool prof_on = c->prof.enabled; c->prof.enabled = false;          // no timing events inside a capture
            Graph g1, g2;
            CUDA_TRY(cudaStreamBeginCapture(ms, cudaStreamCaptureModeThreadLocal));
            rc = enqueue_vg();
            cudaError_t e1 = end_capture(g1, ms);
            if (!rc && e1 == cudaSuccess) {
                CUDA_TRY(cudaStreamBeginCapture(ms, cudaStreamCaptureModeThreadLocal));
                rc = enqueue_grid();
                e1 = end_capture(g2, ms);
            }
            c->prof.enabled = prof_on;
            if (rc || e1 != cudaSuccess) return rc ? rc : LIORF_ERR_CUDA;
            GraphExec vg, grid;                     // the pair is kept only when both instantiate
            CUDA_TRY(graph_instantiate(vg, g1));
            CUDA_TRY(graph_instantiate(grid, g2));
            G.vg = std::move(vg); G.grid = std::move(grid);
            std::memcpy(G.sig, sig, sizeof(sig));
        }
        { ProfScope ps(c, SEC_MAP_BUILD, ms); c->launches += 10; CUDA_TRY(cudaGraphLaunch(G.vg, ms)); }
        { ProfScope ps(c, SEC_GRID_BUILD, ms); c->launches += 3; CUDA_TRY(cudaGraphLaunch(G.grid, ms)); }
    }
    c->m_bound = bound; c->h_m_ds = -1;
    CUDA_TRY(cudaEventRecord(c->ev_map, ms));
    c->map_pending = true;
    c->last_sel = sel; c->last_sel_version = c->pose_version; c->map_valid = true;
    if (m_ds) { if ((rc = read_counts(c))) return rc; *m_ds = c->h_m_ds; return check_err(c); }
    return LIORF_OK;
}

int liorf_extract_nearby(liorf_ctx* c, double time_cur, float density, int* ids, int cap, int* n_ids) {
    LIORF_NVTX;
    if (!c || !ids || !n_ids || cap < 0 || !(density > 0.f)) return LIORF_ERR_ARG;
    std::vector<liorf_host::KeyPose> kp(c->kfs.size());
    for (size_t i = 0; i < kp.size(); ++i) { const Keyframe& k = c->kfs[i]; kp[i] = liorf_host::KeyPose{k.pose[0], k.pose[1], k.pose[2], k.pose[3], k.pose[4], k.pose[5], k.time}; }
    std::vector<int> sel = liorf_host::extract_nearby(kp, time_cur, c->P.surroundingKeyframeSearchRadius, density);
    *n_ids = (int)sel.size();
    if ((int)sel.size() > cap) return LIORF_ERR_ARG;
    std::memcpy(ids, sel.data(), sel.size() * sizeof(int));
    return LIORF_OK;
}
int liorf_save_frame(liorf_ctx* c, const float pose6[6], float dist_thr, float ang_thr) {
    LIORF_NVTX;
    if (!c || !pose6) return LIORF_ERR_ARG;
    if (c->kfs.empty()) return 1;
    const Keyframe& k = c->kfs.back();
    liorf_host::KeyPose last{k.pose[0], k.pose[1], k.pose[2], k.pose[3], k.pose[4], k.pose[5], k.time};
    return liorf_host::save_frame(&last, pose6, dist_thr, ang_thr) ? 1 : 0;
}
void liorf_transform_update_clamp(float pose6[6], float rot_tol, float z_tol) { if (pose6) liorf_host::transform_update_clamp(pose6, rot_tol, z_tol); }
// context-free forms of the same host logic (poses: n x 6 floats (roll,pitch,yaw,x,y,z), times: n doubles)
int liorf_host_extract_nearby(const float* poses6, const double* times, int n, double time_cur, float radius, float density, int* ids, int cap, int* n_ids) {
    if (n < 0 || !n_ids || (n > 0 && (!poses6 || !times)) || !(density > 0.f)) return LIORF_ERR_ARG;
    std::vector<liorf_host::KeyPose> kp(n);
    for (int i = 0; i < n; ++i) kp[i] = liorf_host::KeyPose{poses6[6 * i], poses6[6 * i + 1], poses6[6 * i + 2], poses6[6 * i + 3], poses6[6 * i + 4], poses6[6 * i + 5], times[i]};
    std::vector<int> sel = liorf_host::extract_nearby(kp, time_cur, radius, density);
    *n_ids = (int)sel.size();
    if ((int)sel.size() > cap || !ids) return LIORF_ERR_ARG;
    std::memcpy(ids, sel.data(), sel.size() * sizeof(int));
    return LIORF_OK;
}
static void guess_state_init(liorf_guess_state* st) {
    if (st->initialised) return;
    const float I[12] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0};
    std::memcpy(st->lastImuTransformation, I, sizeof(I)); std::memcpy(st->lastImuPreTransformation, I, sizeof(I));
    st->lastImuPreTransAvailable = 0; st->initialised = 1;
}
int liorf_host_update_initial_guess(liorf_guess_state* state, int no_keyframes_yet, const liorf_cloud_info_guess* ci, int use_imu_heading, int imu_type, float tf[6]) {
    if (!state || !ci || !tf) return LIORF_ERR_ARG;
    guess_state_init(state);
    liorf_host::InitialGuessState s;
    std::memcpy(s.lastImuTransformation, state->lastImuTransformation, 48); std::memcpy(s.lastImuPreTransformation, state->lastImuPreTransformation, 48);
    s.lastImuPreTransAvailable = state->lastImuPreTransAvailable != 0;
    liorf_host::CloudInfoGuess g{ci->imuAvailable, ci->odomAvailable, ci->imuRollInit, ci->imuPitchInit, ci->imuYawInit, ci->initialGuessX, ci->initialGuessY,
                                 ci->initialGuessZ, ci->initialGuessRoll, ci->initialGuessPitch, ci->initialGuessYaw};
    liorf_host::update_initial_guess(s, no_keyframes_yet != 0, g, use_imu_heading != 0, imu_type, tf);
    std::memcpy(state->lastImuTransformation, s.lastImuTransformation, 48); std::memcpy(state->lastImuPreTransformation, s.lastImuPreTransformation, 48);
    state->lastImuPreTransAvailable = s.lastImuPreTransAvailable ? 1 : 0;
    return LIORF_OK;
}
int liorf_host_transform_update(float tf[6], int imu_available, int imu_type, float imu_roll_init, float imu_pitch_init, float imu_rpy_weight, float rot_tol,
                                float z_tol) {
    if (!tf) return LIORF_ERR_ARG;
    liorf_host::transform_update(tf, imu_available != 0, imu_type, imu_roll_init, imu_pitch_init, imu_rpy_weight, rot_tol, z_tol);
    return LIORF_OK;
}
/* ImageProjection::deskewInfo + imuDeskewInfo (src/imageProjection.cpp:330-409): builds the IMU rotation table projectPointCloud reads.
 * Returns 1 = imuAvailable, 0 = table unusable (imuPointerCur <= 0, or the :337 gate said "waiting for IMU data"), negative = error. */
int liorf_host_imu_deskew_info(const double* stamp, const double* gyro_xyz, int n, double time_scan_cur, double time_scan_end, int check_gate,
                               double* imu_time, double* imu_rot_x, double* imu_rot_y, double* imu_rot_z, int capacity, int* imu_pointer_cur, int* n_pop, int* rpy_index) {
    if (n < 0 || (n > 0 && (!stamp || !gyro_xyz)) || !imu_time || !imu_rot_x || !imu_rot_y || !imu_rot_z || capacity < 1 || !imu_pointer_cur) return LIORF_ERR_ARG;
    liorf_host::ImuDeskewInfo info;
    const int rows = liorf_host::imu_deskew_info(stamp, gyro_xyz, n, time_scan_cur, time_scan_end, check_gate != 0, imu_time, imu_rot_x, imu_rot_y, imu_rot_z, capacity, info);
    if (rows == -2) return LIORF_ERR_ARG;
    *imu_pointer_cur = info.imu_pointer_cur;
    if (n_pop) *n_pop = info.n_pop;
    if (rpy_index) *rpy_index = info.rpy_index;
    return info.imu_available ? 1 : 0;
}
int liorf_host_save_frame(const float* last_pose6 /*nullable*/, const float pose6[6], float dist_thr, float ang_thr) {
    if (!pose6) return LIORF_ERR_ARG;
    if (!last_pose6) return 1;
    liorf_host::KeyPose last{last_pose6[0], last_pose6[1], last_pose6[2], last_pose6[3], last_pose6[4], last_pose6[5], 0.0};
    return liorf_host::save_frame(&last, pose6, dist_thr, ang_thr) ? 1 : 0;
}

int liorf_set_local_map(liorf_ctx* c, const liorf_point* map_ds, int m) {
    LIORF_NVTX;
    if (!c || m < 0 || (m > 0 && !map_ds)) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    int rc;
    if ((rc = join_map(c))) return rc;
    if ((rc = c->map_ds.reserve(m > 0 ? m : 1))) return rc;
    if (m > 0) CUDA_TRY(cudaMemcpyAsync(c->map_ds.p, map_ds, (size_t)m * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
    c->h_mail.p[101] = m;
    CUDA_TRY(cudaMemcpyAsync(c->d_shared + C_M_DS, &c->h_mail.p[101], sizeof(int), cudaMemcpyHostToDevice, c->stream));
    c->m_bound = m; c->h_m_ds = m; c->map_valid = false;
    if ((rc = build_map_grid(c->map_ds.p, Count::of_host(m), c->grid, c->stream))) return rc;
    return check_err(c);
}
/* kdtreeSurfFromMap->setInputCloud(laserCloudSurfFromMapDS) (src/mapOptmization.cpp:1302): the reference rebuilds its kd-tree at the top of
 * every scan2MapOptimization call; here the voxel-hash grid is built together with the map (liorf_extract_surrounding_keyframes), so this
 * entry only exists to time / repeat that step on the resident map: asynchronous on the context's stream. */
int liorf_kdtree_set_input_cloud(liorf_ctx* c) {
    LIORF_NVTX;
    if (!c) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    int rc;
    if ((rc = join_map(c))) return rc;
    if (!c->map_ds.p || c->m_bound <= 0) return LIORF_ERR_STATE;
    // on the map stream, like the grid build of liorf_extract_surrounding_keyframes: it runs beside whatever the caller enqueues next on
    // the main stream (downsampleCurrentScan); the solver joins (join_map) before it reads the grid
    if ((rc = need_stream_map(c))) return rc;
    cudaStream_t ms = c->stream_map;
    CUDA_TRY(cudaEventRecord(c->ev_main, c->stream));
    CUDA_TRY(cudaStreamWaitEvent(ms, c->ev_main, 0));
    { ProfScope ps(c, SEC_GRID_BUILD, ms); c->launches += 3; if ((rc = build_map_grid(c->map_ds.p, map_count(c), c->grid, ms))) return rc; }
    CUDA_TRY(cudaEventRecord(c->ev_map, ms));
    c->map_pending = true;
    return LIORF_OK;
}
int liorf_get_local_map(liorf_ctx* c, liorf_point* out, int capacity, int* m_ds) {
    LIORF_NVTX;
    if (!c) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    int rc; if ((rc = read_counts(c))) return rc;
    if (m_ds) *m_ds = c->h_m_ds;
    if (out) { if (capacity < c->h_m_ds) return LIORF_ERR_ARG; if (c->h_m_ds > 0) CUDA_TRY(cudaMemcpy(out, c->map_ds.p, (size_t)c->h_m_ds * sizeof(float4), cudaMemcpyDeviceToHost)); }
    return LIORF_OK;
}
int liorf_get_scan_ds(liorf_ctx* c, liorf_point* out, int capacity, int* n_ds) {
    LIORF_NVTX;
    if (!c) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    int rc; if ((rc = read_counts(c))) return rc;
    if (n_ds) *n_ds = c->h_n_ds;
    if (out) { if (capacity < c->h_n_ds) return LIORF_ERR_ARG; if (c->h_n_ds > 0) CUDA_TRY(cudaMemcpy(out, c->scan_ds.p, (size_t)c->h_n_ds * sizeof(float4), cudaMemcpyDeviceToHost)); }
    return LIORF_OK;
}

static Count scan_ds_count(liorf_ctx* c) { return c->h_n_ds >= 0 ? Count::of_host(c->h_n_ds) : Count::of_dev(c->d_counts + C_N_DS, c->n_scan_bound); }
static Count map_count(liorf_ctx* c) { return c->h_m_ds >= 0 ? Count::of_host(c->h_m_ds) : Count::of_dev(c->d_shared + C_M_DS, c->m_bound); }

// pipelined: the call comes from liorf_process_frame, whose next frame's front end runs beside the solver → leave the spare SMs free
static int launch_s2m(liorf_ctx* c, int max_iters, int force_all, bool pipelined = false, const float* pose6_init = nullptr) {
    if (max_iters < 0) return LIORF_ERR_ARG;
    if (max_iters > S2M_MAX_ITERS) max_iters = S2M_MAX_ITERS;
    c->mail_fresh = false;
    if (!c->grid.cell_start.p || !c->grid.sorted.p) {            // cloudKeyPoses3D empty → return (:1297)
        if (pose6_init) { int rcu = upload_pose(c, pose6_init); if (rcu) return rcu; }
        CUDA_TRY(cudaMemsetAsync(c->d_trace, 0, sizeof(S2MTrace), c->stream));
        return LIORF_OK;
    }
    int rc;
    const size_t qb = (size_t)(c->n_scan_bound > 0 ? c->n_scan_bound : 1);
    if ((rc = c->qcache.reserve(qb)) || (rc = c->cand.reserve(qb * S2M_GROW))) return rc;
    if ((rc = join_map(c))) return rc;
    S2MArgs a;
    a.qcache = c->qcache.p; a.cand = c->cand.p; a.res = c->d_res; a.wpart = c->d_wpart; a.err_flag = c->d_err; a.global_state = c->s2m_global_state ? 1 : 0;
    // epochs of a launch: epoch_base + 1 .. epoch_base + max_iters; they must stay below the next launch's first one, or a worker could
    // take a hand-off word the previous launch left behind for an answer
    static_assert(S2M_MAX_ITERS <= 64, "the epoch stride of the solver launches is 64");
    a.epoch_base = (++c->s2m_launch_seq) * 64u;
    a.scan = c->scan_ds.p; a.n_scan = scan_ds_count(c);
    a.cell_start = c->grid.cell_start.p; a.gmap = c->grid.sorted.p; a.g = c->grid.dims; a.m_map = map_count(c);
    a.tf6 = c->d_tf6; a.st = c->d_lm; a.trace = c->d_trace; a.max_iters = max_iters; a.force_all = force_all; a.no_cache = c->s2m_no_cache ? 1 : 0; a.dbg = c->d_dbg; a.dbg_gt = c->d_dbg_gt;
    a.mail = c->d_mail; a.cnt_n_scan = c->d_counts + C_N_SCAN;
    a.use_tf_init = pose6_init ? 1 : 0;
    for (int k = 0; k < 6; ++k) a.tf_init[k] = pose6_init ? pose6_init[k] : 0.f;
    void* args[] = {&a};
    ProfScope ps(c, SEC_SCAN2MAP); c->launches += 1;
    const int ctas = c->s2m_ctas ? c->s2m_ctas : (pipelined ? c->s2m_grid : c->num_sms);
    CUDA_TRY(cudaLaunchCooperativeKernel((void*)k_scan2map_persistent, dim3(ctas), dim3(S2MP_BLOCK), args, S2MP_SMEM, c->stream));
    c->mail_fresh = true;
    return LIORF_OK;
}

int liorf_scan2map_optimization_async(liorf_ctx* c, const float pose6_in[6], int max_iters, int force_all) {
    LIORF_NVTX;
    if (!c) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    return launch_s2m(c, max_iters, force_all, false, pose6_in);
}
int liorf_get_pose(liorf_ctx* c, float pose6[6], liorf_lm_trace* trace) {
    LIORF_NVTX;
    if (!c || !pose6) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    { int rcj = join_map(c); if (rcj) return rcj; }
    CUDA_TRY(cudaMemcpyAsync(c->h_mail.p + 320, c->d_tf6, 6 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(mail_counts(c));
    if (trace) CUDA_TRY(cudaMemcpyAsync(c->h_mail.p + 1024, c->d_trace, sizeof(S2MTrace), cudaMemcpyDeviceToHost, c->stream));
    else CUDA_TRY(cudaMemcpyAsync(c->h_mail.p + 1024 + 448, &c->d_trace->iters, 4 * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    int rc = check_err(c); if (rc) return rc;
    take_counts(c);                                              // one round trip refreshes the counts too
    c->rep_counts[0] = c->h_n_scan; c->rep_counts[1] = c->h_n_ds; c->rep_counts[2] = c->h_m_ds;
    std::memcpy(pose6, c->h_mail.p + 320, 6 * sizeof(float));
    if (trace) std::memcpy(trace, c->h_mail.p + 1024, sizeof(S2MTrace));
    return LIORF_OK;
}
// liorf_process_frame's round trip: the solver left everything the host needs in ONE 64-byte record (pose, iteration count,
// flags, the three counts, the sticky device error flag) → one D2H copy instead of four.
static int get_pose_mail(liorf_ctx* c, float pose6[6], int* iters, int* converged, int* degenerate, int* ran) {
    if (!c->mail_fresh) {
        int rc = liorf_get_pose(c, pose6, nullptr); if (rc) return rc;
        *iters = c->h_mail.p[1024 + 448]; *converged = c->h_mail.p[1024 + 449]; *degenerate = c->h_mail.p[1024 + 450]; *ran = c->h_mail.p[1024 + 451];
        return LIORF_OK;
    }
    c->mail_fresh = false;
    S2MMail* hm = reinterpret_cast<S2MMail*>(c->h_mail.p + 3200);
    CUDA_TRY(cudaMemcpyAsync(hm, c->d_mail, sizeof(S2MMail), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    prof_flush(c);
    if (hm->err) { fprintf(stderr, "[liorf_b200] device error flag %d (look-back predecessor never arrived)\n", hm->err); return LIORF_ERR_DEVICE_FLAG; }
    std::memcpy(pose6, hm->tf, 6 * sizeof(float));
    *iters = hm->iters; *converged = hm->converged; *degenerate = hm->degenerate; *ran = hm->ran;
    c->h_n_scan = hm->n_scan; c->h_n_ds = hm->n_ds; c->h_m_ds = hm->m_ds;
    c->rep_counts[0] = c->h_n_scan; c->rep_counts[1] = c->h_n_ds; c->rep_counts[2] = c->h_m_ds;
    c->h_mail.p[1024 + 448] = hm->iters;                           // liorf_get_last_counts reads the iteration count here
    return LIORF_OK;
}

int liorf_scan2map_optimization(liorf_ctx* c, float pose6[6], int max_iters, int force_all, liorf_lm_trace* trace) {
    LIORF_NVTX;
    if (!c || !pose6) return LIORF_ERR_ARG;
    int rc = liorf_scan2map_optimization_async(c, pose6, max_iters, force_all);
    if (rc) return rc;
    return liorf_get_pose(c, pose6, trace);
}

int liorf_surf_optimization(liorf_ctx* c, const float pose6[6], liorf_point* coeff, uint8_t* flag, int* nn_idx, float* nn_d2, float* plane,
                            liorf_point* sel) {
    LIORF_NVTX;
    if (!c || !pose6 || !coeff || !flag) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    int rc;
    if (!c->grid.cell_start.p) return LIORF_ERR_STATE;
    if ((rc = join_map(c))) return rc;
    if (c->h_n_ds < 0 && (rc = read_counts(c))) return rc;
    const int n = c->h_n_ds, cap = n > 0 ? n : 1;
    if ((rc = c->h_coeff.reserve(cap)) || (rc = c->h_flag.reserve(cap)) || (rc = c->h_idx.reserve((size_t)5 * cap)) || (rc = c->h_d2.reserve((size_t)5 * cap)) ||
        (rc = c->h_plane.reserve((size_t)4 * cap)) || (rc = c->h_sel_pts.reserve(cap))) return rc;
    if ((rc = upload_pose(c, pose6))) return rc;
    c->hook_n = n;
    if (n > 0) {
        k_surf_optimization<<<(n + S2M_QPB - 1) / S2M_QPB, S2M_BLOCK, 0, c->stream>>>(c->scan_ds.p, Count::of_host(n), c->d_tf6, c->grid.cell_start.p,
            c->grid.sorted.p, c->grid.dims, map_count(c), c->h_coeff.p, c->h_flag.p, c->h_idx.p, c->h_d2.p, c->h_plane.p, c->h_sel_pts.p);
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaMemcpyAsync(coeff, c->h_coeff.p, (size_t)n * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(cudaMemcpyAsync(flag, c->h_flag.p, (size_t)n, cudaMemcpyDeviceToHost, c->stream));
        if (nn_idx) CUDA_TRY(cudaMemcpyAsync(nn_idx, c->h_idx.p, (size_t)5 * n * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        if (nn_d2) CUDA_TRY(cudaMemcpyAsync(nn_d2, c->h_d2.p, (size_t)5 * n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
        if (plane) CUDA_TRY(cudaMemcpyAsync(plane, c->h_plane.p, (size_t)4 * n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
        if (sel) CUDA_TRY(cudaMemcpyAsync(sel, c->h_sel_pts.p, (size_t)n * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
    }
    return check_err(c);
}

int liorf_combine_optimization_coeffs(liorf_ctx* c, liorf_point* ori, liorf_point* coeff, int* n_sel) {
    LIORF_NVTX;
    if (!c || !n_sel) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    int rc; const int n = c->hook_n, cap = n > 0 ? n : 1;
    if ((rc = c->h_ori_c.reserve(cap)) || (rc = c->h_coeff_c.reserve(cap))) return rc;
    if ((rc = launch_scan(Count::of_host(n), FlagLoad{c->h_flag.p}, CombineStore{c->scan_ds.p, c->h_coeff.p, c->h_ori_c.p, c->h_coeff_c.p}, c->combine_scan,
                          (unsigned*)(c->d_counts + C_HOOK_NSEL), c->stream))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->h_mail.p + 400, c->d_counts + C_HOOK_NSEL, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    const int ns = c->h_mail.p[400]; *n_sel = ns;
    if (ori && ns > 0) CUDA_TRY(cudaMemcpyAsync(ori, c->h_ori_c.p, (size_t)ns * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
    if (coeff && ns > 0) CUDA_TRY(cudaMemcpyAsync(coeff, c->h_coeff_c.p, (size_t)ns * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
    return check_err(c);
}

int liorf_lm_optimization(liorf_ctx* c, int iter, float pose6[6], float AtA[36], float AtB[6], float X[6], int* n_sel) {
    LIORF_NVTX;
    if (!c || !pose6) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    int rc; const int nb = c->hook_n > 0 ? c->hook_n : 1;
    int blocks = (nb + 255) / 256; if (blocks > 2 * c->num_sms) blocks = 2 * c->num_sms;
    if ((rc = c->lm_partial.reserve((size_t)blocks * NPROD))) return rc;
    if ((rc = upload_pose(c, pose6))) return rc;
    k_lm_hook<<<blocks, 256, 0, c->stream>>>(iter, c->h_ori_c.p, c->h_coeff_c.p, (const unsigned*)(c->d_counts + C_HOOK_NSEL), c->d_tf6, c->d_lm,
                                             c->lm_partial.p, c->d_misc + 7, c->d_lm_out, c->d_lm_out + 36, c->d_lm_out + 42, c->d_counts + C_NSEL,
                                             c->d_counts + C_CONV);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(c->h_mail.p + 320, c->d_tf6, 6 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(c->h_mail.p + 500, c->d_lm_out, 48 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(c->h_mail.p + 600, c->d_counts, C_COUNT * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    if ((rc = check_err(c))) return rc;
    std::memcpy(pose6, c->h_mail.p + 320, 6 * sizeof(float));
    const float* o = reinterpret_cast<const float*>(c->h_mail.p + 500);
    if (AtA) std::memcpy(AtA, o, 36 * sizeof(float));
    if (AtB) std::memcpy(AtB, o + 36, 6 * sizeof(float));
    if (X) std::memcpy(X, o + 42, 6 * sizeof(float));
    if (n_sel) *n_sel = c->h_mail.p[600 + C_NSEL];
    return c->h_mail.p[600 + C_CONV] ? 1 : 0;
}
int liorf_get_lm_state(liorf_ctx* c, int* deg, float matP[36]) {
    LIORF_NVTX;
    if (!c) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    LMDeviceState s; CUDA_TRY(cudaStreamSynchronize(c->stream));
    CUDA_TRY(cudaMemcpy(&s, c->d_lm, sizeof(s), cudaMemcpyDeviceToHost));
    if (deg) *deg = s.isDegenerate; if (matP) std::memcpy(matP, s.matP, sizeof(s.matP));
    return LIORF_OK;
}
int liorf_set_lm_state(liorf_ctx* c, int deg, const float matP[36]) {
    LIORF_NVTX;
    if (!c || !matP) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    LMDeviceState s; s.isDegenerate = deg; std::memcpy(s.matP, matP, sizeof(s.matP));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    CUDA_TRY(cudaMemcpy(c->d_lm, &s, sizeof(s), cudaMemcpyHostToDevice));
    return LIORF_OK;
}

// ------------------------------------------------------------------------------------------------ ScanContext
int liorf_sc_make_and_save(liorf_ctx* c, const liorf_point* cloud, int n) {
    LIORF_NVTX;
    if (!c) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    int rc;
    const float4* d_pts; Count cnt = Count::of_host(0);
    if (cloud) {
        if (n < 0) return LIORF_ERR_ARG;
        if ((rc = join_map(c))) return rc;
        if ((rc = c->map_raw.reserve(n > 0 ? n : 1))) return rc;
        c->map_valid = false;
        if (n > 0) CUDA_TRY(cudaMemcpyAsync(c->map_raw.p, cloud, (size_t)n * sizeof(float4), cudaMemcpyHostToDevice, c->stream));
        d_pts = c->map_raw.p; cnt = Count::of_host(n);
    } else {
        d_pts = c->scan.p; cnt = c->h_n_scan >= 0 ? Count::of_host(c->h_n_scan) : Count::of_dev(c->d_counts + C_N_SCAN, c->n_scan_bound);
    }
    if (c->sc_borrowed()) return LIORF_ERR_STATE;
    if ((rc = sc_reserve(c, c->sc_n + 1))) return rc;
    ProfScope ps(c, SEC_SC_MAKE); c->launches += 2;
    if (cnt.bound > 0) {
        int blocks = (cnt.bound + 256 * 8 - 1) / (256 * 8); if (blocks > c->num_sms) blocks = c->num_sms;
        k_sc_bins<<<blocks, 256, 0, c->stream>>>(d_pts, cnt, c->d_bins);
    }
    const size_t e = (size_t)c->sc_n;
    k_sc_finalize<<<1, 64, 0, c->stream>>>(c->d_bins, nullptr, c->sc_db->desc.p + e * SC_DESC, c->sc_db->keys.p + e * SC_RING, c->sc_db->sk.p + e * SC_SECTOR,
                                           c->sc_db->cn.p + e * SC_SECTOR);
    CUDA_TRY(cudaGetLastError());
    ++c->sc_n;
    if (cloud) CUDA_TRY(cudaStreamSynchronize(c->stream));
    return LIORF_OK;
}

int liorf_sc_add_descriptors(liorf_ctx* c, const double* descs, int count) {
    LIORF_NVTX;
    if (!c || count < 0 || (count > 0 && !descs)) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    int rc;
    if (count == 0) return LIORF_OK;
    if (c->sc_borrowed()) return LIORF_ERR_STATE;
    if ((rc = sc_reserve(c, c->sc_n + count))) return rc;
    const size_t e = (size_t)c->sc_n;
    CUDA_TRY(cudaMemcpyAsync(c->sc_db->desc.p + e * SC_DESC, descs, (size_t)count * SC_DESC * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    k_sc_keys_batch<<<count, 64, 0, c->stream>>>(c->sc_db->desc.p + e * SC_DESC, count, c->sc_db->keys.p + e * SC_RING, c->sc_db->sk.p + e * SC_SECTOR,
                                                 c->sc_db->cn.p + e * SC_SECTOR);
    CUDA_TRY(cudaGetLastError());
    c->sc_n += count;
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return LIORF_OK;
}
/* A second context on the same device that searches the SAME database (descriptors, ring keys, sector keys, column norms are not copied):
 * several query batches in flight on one GPU, each on its own context / stream.  The borrower never adds entries; the owner must outlive it
 * and must not grow the database while it is borrowed. */
int liorf_sc_borrow_database(liorf_ctx* dst, liorf_ctx* src) {
    LIORF_NVTX;
    if (!dst || !src || dst == src || dst->P.device != src->P.device) return LIORF_ERR_ARG;
    if (!dst->sc_borrowed() && (dst->sc_n != 0 || dst->sc_own.desc.p)) return LIORF_ERR_STATE;
    CUDA_TRY(cudaSetDevice(src->P.device));
    CUDA_TRY(cudaStreamSynchronize(src->stream));
    dst->sc_db = src->sc_db; dst->sc_n = src->sc_n;            // borrowing from a borrower reads the owner's database
    // a sharded owner's replicated index (liorf_sc_shard_sync_keys) is shared too; the borrower builds its own operand image from it
    dst->ks_all.keys = src->ks_all.keys; dst->ks_all.n = src->ks_all.n; dst->ks_all.gen = src->ks_all.gen;
    return LIORF_OK;
}
int liorf_sc_size(liorf_ctx* c) { return c ? c->sc_n : LIORF_ERR_ARG; }
int liorf_sc_get(liorf_ctx* c, int i, double desc[1200], float ringkey[20], double sectorkey[60]) {
    LIORF_NVTX;
    if (!c || i < 0 || i >= c->sc_n) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    if (desc) CUDA_TRY(cudaMemcpy(desc, c->sc_db->desc.p + (size_t)i * SC_DESC, SC_DESC * sizeof(double), cudaMemcpyDeviceToHost));
    if (ringkey) CUDA_TRY(cudaMemcpy(ringkey, c->sc_db->keys.p + (size_t)i * SC_RING, SC_RING * sizeof(float), cudaMemcpyDeviceToHost));
    if (sectorkey) CUDA_TRY(cudaMemcpy(sectorkey, c->sc_db->sk.p + (size_t)i * SC_SECTOR, SC_SECTOR * sizeof(double), cudaMemcpyDeviceToHost));
    return LIORF_OK;
}

// local exact top-3 of Q queries over keys[0:n_keys) → d_dist/d_idx [Q][3]; unfilled slots: dist +inf, idx INT_MAX
// lim (nullable, device [Q]): query q sees only keys [0, lim[q]) (every lim[q] <= n_keys)
static int sc_knn_brute(liorf_ctx* c, const float* d_keys, int n_keys, const float* d_qkeys, int Q, int global_offset, float* d_dist, int* d_idx,
                        const int* lim = nullptr) {
    int rc;
    if (Q <= 0) return LIORF_OK;
    const int bx = (Q + SCK_BLOCK - 1) / SCK_BLOCK;
    int max_chunks = (n_keys + SCK_TILE - 1) / SCK_TILE; if (max_chunks < 1) max_chunks = 1;
    int chunks = (4 * c->num_sms + bx - 1) / bx; if (chunks > max_chunks) chunks = max_chunks; if (chunks < 1) chunks = 1;
    int kpc = (n_keys + chunks - 1) / chunks; kpc = ((kpc + SCK_TILE - 1) / SCK_TILE) * SCK_TILE; if (kpc < SCK_TILE) kpc = SCK_TILE;
    chunks = (n_keys + kpc - 1) / kpc; if (chunks < 1) chunks = 1;
    if ((rc = c->sc_part_d.reserve((size_t)chunks * Q * 3)) || (rc = c->sc_part_i.reserve((size_t)chunks * Q * 3))) return rc;
    ProfScope ps(c, SEC_SC_SEARCH); c->launches += 2;
    if (lim) k_sc_knn_tile<true><<<dim3(bx, chunks), SCK_BLOCK, 0, c->stream>>>(d_keys, n_keys, global_offset, d_qkeys, Q, kpc, c->sc_part_d.p, c->sc_part_i.p, lim);
    else k_sc_knn_tile<false><<<dim3(bx, chunks), SCK_BLOCK, 0, c->stream>>>(d_keys, n_keys, global_offset, d_qkeys, Q, kpc, c->sc_part_d.p, c->sc_part_i.p, nullptr);
    k_sc_merge_top3<<<(Q + 127) / 128, 128, 0, c->stream>>>(c->sc_part_d.p, c->sc_part_i.p, chunks, (size_t)Q * 3, Q, d_dist, d_idx);
    CUDA_TRY(cudaGetLastError());
    return LIORF_OK;
}

// tensor-core path (sc_tensor.cuh): operand images → GEMM filter → thresholds → candidates → exact re-rank.
// The B image of a key set is rebuilt only when the set changed since it was made.
static int sct_prepare(liorf_ctx* c, liorf_ctx::KeySet& ks, int n_keys, const float* d_qkeys, int Q, SctArgs& a, int& grid) {
    int rc;
    const int nkt = (n_keys + SCT_KT - 1) / SCT_KT, n_sqt = (Q + SCT_QT - 1) / SCT_QT;
    if (!ks.center) CUDA_TRY(dev_alloc(ks.center, SC_RING));
    if (!ks.nmax) CUDA_TRY(dev_alloc(ks.nmax, 1));
    if (!c->sct_over_cnt) { CUDA_TRY(dev_alloc(c->sct_over_cnt, 1)); CUDA_TRY(cudaMemsetAsync(c->sct_over_cnt, 0, sizeof(int), c->stream)); }
    if (!c->sct_attr_set) {
        CUDA_TRY(cudaFuncSetAttribute(k_sc_tensor<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SCT_SMEM));
        CUDA_TRY(cudaFuncSetAttribute(k_sc_tensor<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SCT_SMEM));
        CUDA_TRY(cudaFuncSetAttribute(k_sc_tensor<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SCT_SMEM));
        c->sct_attr_set = true;
    }
    if (ks.img_n != n_keys || ks.img_gen != ks.gen || ks.img_keys != ks.keys) {
        if ((rc = ks.bimg.reserve((size_t)nkt * SCT_TILE_BYTES))) return rc;
        k_sct_center<<<1, 1024, 0, c->stream>>>(ks.keys, n_keys, ks.center);
        CUDA_TRY(cudaMemsetAsync(ks.nmax, 0, sizeof(unsigned), c->stream));
        k_sct_image<true><<<(nkt * SCT_KT + 127) / 128, 128, 0, c->stream>>>(ks.keys, n_keys, nkt * SCT_KT, nkt, ks.center, ks.bimg.p, nullptr, ks.nmax);
        CUDA_TRY(cudaGetLastError());
        ks.img_n = n_keys; ks.img_gen = ks.gen; ks.img_keys = ks.keys; c->launches += 2;
    }
    const long long total = (long long)n_sqt * nkt;
    grid = (int)(total < c->num_sms ? total : c->num_sms);
    const size_t rows = (size_t)n_sqt * SCT_QT;
    if ((rc = c->sct_aimg.reserve((size_t)n_sqt * 2 * SCT_TILE_BYTES)) || (rc = c->sct_qnorm.reserve(rows)) || (rc = c->sct_cmin.reserve(rows * nkt)) || (rc = c->sct_cmin32.reserve(rows * nkt * 4)) || (rc = c->sct_part.reserve(rows * SCS_SPLITS * 3)) ||
        (rc = c->sct_cand.reserve((size_t)Q * SCT_CAP)) || (rc = c->sct_cnt.reserve(Q))) return rc;
    k_sct_image<false><<<(int)((rows + 127) / 128), 128, 0, c->stream>>>(d_qkeys, Q, (int)rows, nkt, ks.center, c->sct_aimg.p, c->sct_qnorm.p, nullptr);
    a.a_img = c->sct_aimg.p; a.b_img = ks.bimg.p; a.Q = Q; a.n_keys = n_keys; a.nkt = nkt; a.n_sqt = n_sqt;
    a.cmin = c->sct_cmin.p; a.cmin32 = c->sct_cmin32.p; a.dump = nullptr; a.err_flag = c->d_err; a.lim = nullptr;
    c->launches += 1;
    return LIORF_OK;
}

// exact top-3 of Q queries over the first n_keys keys of a key set on the tensor cores.  push != nullptr: sharded search, the result goes
// into every rank's window (phase C) from the re-rank kernel itself.  lim (nullable, device [Q]): query q sees only keys [0, lim[q]); the
// filter still runs over the operand image of all n_keys keys, so the cached image is reused whatever the limits
static int sc_knn_tensor(liorf_ctx* c, liorf_ctx::KeySet& ks, int n_keys, const float* d_qkeys, int Q, int idx_offset, float* d_dist, int* d_idx, const ShardPush* push = nullptr,
                         const int* lim = nullptr) {
    int rc, grid;
    SctArgs a;
    ProfScope ps(c, SEC_SC_SEARCH);
    const int nkt = (n_keys + SCT_KT - 1) / SCT_KT, rows = ((Q + SCT_QT - 1) / SCT_QT) * SCT_QT;
    if ((rc = sct_prepare(c, ks, n_keys, d_qkeys, Q, a, grid))) return rc;
    a.lim = lim;
    {
        ProfScope pg(c, SEC_SC_GEMM);
        if (lim) k_sc_tensor<false, true><<<grid, SCT_THREADS, SCT_SMEM, c->stream>>>(a);
        else k_sc_tensor<false><<<grid, SCT_THREADS, SCT_SMEM, c->stream>>>(a);
    }
    k_sct_top3<<<dim3(rows / 32, SCS_SPLITS), 32 * SCS_SLICES, 0, c->stream>>>(c->sct_cmin.p, nkt, rows, c->sct_part.p, Q, c->sct_cnt.p, c->sct_over_cnt);
    k_sct_select<<<dim3(rows / 32, SCS_SPLITS), 32 * SCS_SLICES, 0, c->stream>>>(c->sct_cmin.p, c->sct_cmin32.p, nkt, rows, c->sct_part.p, c->sct_qnorm.p, Q, ks.nmax,
                                                                                 c->sct_cand.p, c->sct_cnt.p);
    ShardPush P; std::memset(&P, 0, sizeof(P));
    if (push) P = *push;
    if (lim) k_sct_rerank<true><<<(Q + 7) / 8, 256, 0, c->stream>>>(ks.keys, n_keys, nkt, idx_offset, d_qkeys, Q, c->sct_cand.p, c->sct_cnt.p, d_dist, d_idx, c->sct_over_cnt, P, lim);
    else k_sct_rerank<false><<<(Q + 7) / 8, 256, 0, c->stream>>>(ks.keys, n_keys, nkt, idx_offset, d_qkeys, Q, c->sct_cand.p, c->sct_cnt.p, d_dist, d_idx, c->sct_over_cnt, P, nullptr);
    CUDA_TRY(cudaGetLastError());
    c->launches += 4; c->sct_last_Q = Q;
    return LIORF_OK;
}

static bool sc_want_tensor(const liorf_ctx* c, int Q, int n_keys) {
    // the tensor-core filter pays off for query batches against a sizeable database; the live detectLoopClosureID (one query) stays on the
    // exact CUDA-core kernel
    return n_keys >= 1 && (c->sc_path == 2 || (c->sc_path == 0 && Q >= 64 && n_keys >= 4096));
}
static int sc_knn(liorf_ctx* c, liorf_ctx::KeySet& ks, int n_keys, const float* d_qkeys, int Q, int idx_offset, float* d_dist, int* d_idx) {
    if (Q <= 0) return LIORF_OK;
    if (sc_want_tensor(c, Q, n_keys)) return sc_knn_tensor(c, ks, n_keys, d_qkeys, Q, idx_offset, d_dist, d_idx);
    return sc_knn_brute(c, ks.keys, n_keys, d_qkeys, Q, idx_offset, d_dist, d_idx);
}
static liorf_ctx::KeySet& local_keys(liorf_ctx* c) { c->ks_local.keys = c->sc_db->keys.p; c->ks_local.n = c->sc_n; return c->ks_local; }

// shared-memory limit and occupancy of both instantiations of the stage-2 kernel, once per context
static int scdb_setup(liorf_ctx* c) {
    if (c->scdb_attr_set) return LIORF_OK;
    int occ = 0;
    CUDA_TRY(cudaFuncSetAttribute(k_sc_distance_bulk<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SCDB_SMEM));
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_sc_distance_bulk<false>, SCDB_THREADS, SCDB_SMEM));
    c->scdb_blocks_per_sm[0] = occ > 0 ? occ : 1;
    CUDA_TRY(cudaFuncSetAttribute(k_sc_distance_bulk<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SCDB_SMEM));
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_sc_distance_bulk<true>, SCDB_THREADS, SCDB_SMEM));
    c->scdb_blocks_per_sm[1] = occ > 0 ? occ : 1;
    c->scdb_attr_set = true;
    return LIORF_OK;
}

// stage 2 for a batch of (query, candidate) pairs: TMA-staged kernel (sc_distance.cuh), persistent warps over the pairs.
// Query descriptors need only 8-byte alignment: a 16-byte-aligned array takes the kernel's 16-byte loads, any other the scalar-load
// instantiation (same results).  Every launch of k_sc_distance_bulk goes through here.
static int sc_distance_launch(liorf_ctx* c, const double* qd, const int* cand, int pairs, int global_offset, double* pd, int* ps,
                              const int* pair_list = nullptr, const int* n_list = nullptr, const ShardPush* push = nullptr) {
    int rc;
    if ((rc = scdb_setup(c))) return rc;
    const bool q16 = ((uintptr_t)qd & 15) == 0;
    // persistent warps, one pair at a time each: the fewest CTAs that still finish in the same number of rounds (a sharded rank owns
    // about pairs / world of the pairs: 5.2 rounds of the full grid are 6 rounds either way, and the CTAs not launched leave their
    // shared memory to the other lanes' kernels)
    const int cap = c->num_sms * c->scdb_blocks_per_sm[q16];
    const long long est = push ? ((long long)pairs + push->W.world - 1) / push->W.world : pairs;
    const long long rounds = std::max<long long>(1, (est + (long long)cap * SCDB_WARPS - 1) / ((long long)cap * SCDB_WARPS));
    int blocks = (int)((est + rounds * SCDB_WARPS - 1) / (rounds * SCDB_WARPS));
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;                                   // a rank that owns no pair still raises its phase-D flag
    ShardPush P; std::memset(&P, 0, sizeof(P));
    if (push) P = *push;
    if (q16) k_sc_distance_bulk<true><<<blocks, SCDB_THREADS, SCDB_SMEM, c->stream>>>(qd, cand, pairs, SC_NUM_CAND, c->sc_db->desc.p, c->sc_db->sk.p, c->sc_db->cn.p, global_offset,
                                                                                    c->sc_n, pd, ps, c->d_err, pair_list, n_list, P);
    else k_sc_distance_bulk<false><<<blocks, SCDB_THREADS, SCDB_SMEM, c->stream>>>(qd, cand, pairs, SC_NUM_CAND, c->sc_db->desc.p, c->sc_db->sk.p, c->sc_db->cn.p, global_offset,
                                                                                 c->sc_n, pd, ps, c->d_err, pair_list, n_list, P);
    CUDA_TRY(cudaGetLastError());
    c->launches += 1;
    return LIORF_OK;
}

int liorf_sc_knn_batch_dev(liorf_ctx* c, const void* d_qkeys, int Q, int global_offset, void* d_dist, void* d_idx) {
    LIORF_NVTX;
    if (!c || Q < 0 || !d_qkeys || !d_dist || !d_idx) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    return sc_knn(c, local_keys(c), c->sc_n, (const float*)d_qkeys, Q, global_offset, (float*)d_dist, (int*)d_idx);
}
int liorf_sc_prepare_queries_dev(liorf_ctx* c, const void* d_qdescs, int Q, void* d_qkeys, void* d_qsk, void* d_qcn) {
    LIORF_NVTX;
    if (!c || Q < 0 || !d_qdescs || (!d_qkeys && !d_qsk)) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    if (Q == 0) return LIORF_OK;
    if (d_qkeys && !d_qsk && ((uintptr_t)d_qdescs & 15) == 0) k_sc_ringkeys_batch<<<(Q + SCK_WARPS - 1) / SCK_WARPS, 32 * SCK_WARPS, 0, c->stream>>>((const double*)d_qdescs, Q, (float*)d_qkeys);
    else k_sc_keys_batch<<<Q, 64, 0, c->stream>>>((const double*)d_qdescs, Q, (float*)d_qkeys, (double*)d_qsk, (double*)d_qcn);
    CUDA_TRY(cudaGetLastError());
    c->launches += 1;
    return LIORF_OK;
}
int liorf_sc_distance_batch_dev(liorf_ctx* c, const void* d_qdescs, const void* d_cand_idx, int Q, int global_offset, void* d_pair_dist, void* d_pair_shift) {
    LIORF_NVTX;
    if (!c || Q < 0 || !d_qdescs || !d_cand_idx || !d_pair_dist || !d_pair_shift) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    if (Q == 0) return LIORF_OK;
    return sc_distance_launch(c, (const double*)d_qdescs, (const int*)d_cand_idx, Q * SC_NUM_CAND, global_offset, (double*)d_pair_dist, (int*)d_pair_shift);
}
int liorf_sc_decide_dev(liorf_ctx* c, const void* d_pair_dist, const void* d_pair_shift, const void* d_cand_idx, int Q, void* d_loop_id, void* d_shift,
                        void* d_dist) {
    LIORF_NVTX;
    if (!c || Q < 0) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    if (Q == 0) return LIORF_OK;
    k_sc_decide<<<(Q + 127) / 128, 128, 0, c->stream>>>((const double*)d_pair_dist, (const int*)d_pair_shift, (const int*)d_cand_idx, Q, (int*)d_loop_id,
                                                         (int*)d_shift, (double*)d_dist);
    CUDA_TRY(cudaGetLastError());
    c->launches += 1;
    return LIORF_OK;
}

/* tests: the stage-2 grid bound: SMs and CTAs per SM of the 16-byte-aligned and the 8-byte-aligned query instantiations */
int liorf_debug_sc_distance_occupancy(liorf_ctx* c, int out[3]) {
    LIORF_NVTX;
    if (!c || !out) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    int rc;
    if ((rc = scdb_setup(c))) return rc;
    out[0] = c->num_sms; out[1] = c->scdb_blocks_per_sm[1]; out[2] = c->scdb_blocks_per_sm[0];
    return LIORF_OK;
}

/* tests: cv::solve(DECOMP_QR) (hal::QR32f) of n 6x6 systems (A row-major [n][36], b [n][6]) by the device routine of the solver */
int liorf_debug_qr_solve6(liorf_ctx* c, const float* A, const float* b, int n, float* x) {
    LIORF_NVTX;
    if (!c || !A || !b || n <= 0 || !x) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    DevBuf<float> d; int rc;
    if ((rc = d.reserve((size_t)n * (36 + 6 + 6)))) return rc;
    float* dA = d.p; float* db = dA + (size_t)36 * n; float* dx = db + (size_t)6 * n;
    CUDA_TRY(cudaMemcpyAsync(dA, A, (size_t)36 * n * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaMemcpyAsync(db, b, (size_t)6 * n * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    k_debug_qr6<<<(n + 1) / 2, 64, 0, c->stream>>>(dA, db, n, dx, c->d_err);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(x, dx, (size_t)6 * n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    return check_err(c);
}
/* tests: 1 = run the multi-kernel (large-cloud) VoxelGrid path on small clouds too; 0 = automatic */
int liorf_debug_force_large_voxelgrid(liorf_ctx* c, int on) {
    LIORF_NVTX;
    if (!c) return LIORF_ERR_ARG;
    c->vg.force_large = c->vg_map.force_large = c->alt.vg.force_large = on != 0;
    c->vg.force_multi = c->vg_map.force_multi = c->alt.vg.force_multi = on != 0;
    return LIORF_OK;
}
/* debug: %globaltimer stamps (ns) of CTA 0 at the phase boundaries of the last one-kernel VoxelGrid of the scan side */
int liorf_debug_voxelgrid_stamps(liorf_ctx* c, int enable, unsigned long long* out /* 32, nullable */) {
    LIORF_NVTX;
    if (!c) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    if (enable && !c->vg.dbg) { CUDA_TRY(dev_alloc(c->vg.dbg, 32)); CUDA_TRY(cudaMemset(c->vg.dbg, 0, 32 * sizeof(unsigned long long))); }
    if (out && c->vg.dbg) CUDA_TRY(cudaMemcpy(out, c->vg.dbg, 32 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    if (!enable) c->vg.dbg.reset();
    return LIORF_OK;
}
/* tests: 1 = run the one-kernel cooperative VoxelGrid path on small clouds too; 0 = automatic */
int liorf_debug_force_fused_voxelgrid(liorf_ctx* c, int on) {
    LIORF_NVTX;
    if (!c) return LIORF_ERR_ARG;
    c->vg.force_large = c->vg_map.force_large = c->alt.vg.force_large = on != 0;
    c->vg.force_multi = c->vg_map.force_multi = c->alt.vg.force_multi = false;
    return LIORF_OK;
}
/* tests: liorf_voxel_grid runs the one-kernel cooperative VoxelGrid on `ctas` CTAs (0 = all SMs), so that every chunk length and grid width
 * it can run with is reachable from small clouds.  Its grid barrier needs every CTA resident at once: widths beyond what the device holds
 * co-resident are refused. */
int liorf_debug_voxelgrid_grid(liorf_ctx* c, int ctas) {
    LIORF_NVTX;
    if (!c || ctas < 0) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    int occ = 0;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_vg_fused, VGF_THREADS, 0));
    if (ctas > occ * c->num_sms) return LIORF_ERR_ARG;
    c->vg_ctas = ctas;
    return LIORF_OK;
}
/* selects the ring-key search implementation: 0 auto, 1 CUDA-core brute force, 2 tensor-core filter + exact re-rank */
int liorf_sc_set_search_path(liorf_ctx* c, int mode) {
    LIORF_NVTX;
    if (!c || mode < 0 || mode > 2) return LIORF_ERR_ARG;
    c->sc_path = mode;
    return LIORF_OK;
}
/* statistics of the last tensor-core search: candidates emitted by the coarse filter (sum over queries), queries that
 * overflowed their list and were answered by the exact scan instead */
int liorf_sc_tensor_stats(liorf_ctx* c, long long* n_candidates, int* n_overflow) {
    LIORF_NVTX;
    if (!c || !n_candidates || !n_overflow) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    *n_candidates = 0; *n_overflow = 0;
    const int Q = c->sct_last_Q;
    if (Q <= 0 || !c->sct_cnt.p) return LIORF_OK;
    std::vector<int> cnt(Q);
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    CUDA_TRY(cudaMemcpy(cnt.data(), c->sct_cnt.p, (size_t)Q * sizeof(int), cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(n_overflow, c->sct_over_cnt, sizeof(int), cudaMemcpyDeviceToHost));
    for (int v : cnt) *n_candidates += v;
    return LIORF_OK;
}
/* test hook: the raw tensor-core distances d~ of Q host queries (ring keys) against the whole database,
 * out[(q) * ld + k] with ld = ceil(n_db / 128) * 128 (returned), center[20] = the database mean the images use */
int liorf_sc_tensor_dump(liorf_ctx* c, const float* qkeys, int Q, float* out, long long out_capacity, int* ld, float center[20]) {
    LIORF_NVTX;
    if (!c || !qkeys || Q <= 0 || !out || !ld) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    if (c->sc_n < 1) return LIORF_ERR_STATE;
    int rc, grid;
    if ((rc = c->sc_qkeys.reserve((size_t)Q * SC_RING))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->sc_qkeys.p, qkeys, (size_t)Q * SC_RING * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    SctArgs a;
    liorf_ctx::KeySet& ks = local_keys(c);
    if ((rc = sct_prepare(c, ks, c->sc_n, c->sc_qkeys.p, Q, a, grid))) return rc;
    const size_t rows = (size_t)a.n_sqt * SCT_QT, cols = (size_t)a.nkt * SCT_KT;
    *ld = (int)cols;
    if ((long long)((size_t)Q * cols) > out_capacity) return LIORF_ERR_ARG;
    DevBuf<float> dump; if ((rc = dump.reserve(rows * cols))) return rc;
    a.dump = dump.p;
    k_sc_tensor<true><<<grid, SCT_THREADS, SCT_SMEM, c->stream>>>(a);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(out, dump.p, (size_t)Q * cols * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    if (center) CUDA_TRY(cudaMemcpyAsync(center, ks.center, SC_RING * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    return check_err(c);
}

static int sc_reserve_query(liorf_ctx* c, int Q) {
    int rc;
    if ((rc = c->sc_q_d.reserve((size_t)3 * Q)) || (rc = c->sc_q_i.reserve((size_t)3 * Q)) || (rc = c->sc_pair_d.reserve((size_t)3 * Q)) ||
        (rc = c->sc_pair_s.reserve((size_t)3 * Q)) || (rc = c->sc_res_i.reserve((size_t)2 * Q)) || (rc = c->sc_res_d.reserve(Q))) return rc;
    return LIORF_OK;
}

// the unsharded batch on device buffers: ring keys of the queries → exact top-3 → distanceBtnScanContext of the 3 Q pairs → decision
static int sc_query_local_dev(liorf_ctx* c, const double* qd, int Q, int global_offset, int* cand, int* d_loop_id, int* d_shift, double* d_dist) {
    int rc;
    if ((rc = c->sc_qkeys.reserve((size_t)Q * SC_RING)) || (rc = sc_reserve_query(c, Q))) return rc;
    if ((rc = liorf_sc_prepare_queries_dev(c, qd, Q, c->sc_qkeys.p, nullptr, nullptr))) return rc;
    if ((rc = sc_knn(c, local_keys(c), c->sc_n, c->sc_qkeys.p, Q, global_offset, c->sc_q_d.p, cand))) return rc;
    if ((rc = sc_distance_launch(c, qd, cand, 3 * Q, global_offset, c->sc_pair_d.p, c->sc_pair_s.p))) return rc;
    return liorf_sc_decide_dev(c, c->sc_pair_d.p, c->sc_pair_s.p, cand, Q, d_loop_id, d_shift, d_dist);
}

int liorf_sc_query_batch(liorf_ctx* c, const double* qdescs, int Q, int* loop_id, int* shift, double* dist, int* cand3) {
    LIORF_NVTX;
    if (!c || Q < 0 || (Q > 0 && (!qdescs || !loop_id || !shift || !dist))) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    if (Q == 0) return LIORF_OK;
    if (c->sc_n < 1) return LIORF_ERR_STATE;
    int rc;
    if ((rc = c->sc_qdesc.reserve((size_t)Q * SC_DESC)) || (rc = sc_reserve_query(c, Q))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->sc_qdesc.p, qdescs, (size_t)Q * SC_DESC * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    if ((rc = sc_query_local_dev(c, c->sc_qdesc.p, Q, 0, c->sc_q_i.p, c->sc_res_i.p, c->sc_res_i.p + Q, c->sc_res_d.p))) return rc;
    CUDA_TRY(cudaMemcpyAsync(loop_id, c->sc_res_i.p, (size_t)Q * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(shift, c->sc_res_i.p + Q, (size_t)Q * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(dist, c->sc_res_d.p, (size_t)Q * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    if (cand3) CUDA_TRY(cudaMemcpyAsync(cand3, c->sc_q_i.p, (size_t)3 * Q * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    return check_err(c);
}

// ---- sharded search over NVLink peer windows (sc_shard.cuh) ----
static size_t scsh_round(size_t b) { return (b + 255) / 256 * 256; }
int liorf_sc_shard_init(liorf_ctx* c, int rank, int world, int q_max, int k_total_max, void* ipc_handle_out /*64 B, nullable*/, void** window_out /*nullable*/) {
    LIORF_NVTX;
    if (!c || world < 1 || world > SCSH_MAX || rank < 0 || rank >= world || q_max < 1 || k_total_max < 0) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    liorf_ctx::ScShard& S = c->shard;
    if (S.ready || S.W.base[S.W.rank]) return LIORF_ERR_STATE;
    if (world > 1) {   // see need_stream_map: consumer kernels of different lanes wait for flags of OTHER GPUs; their streams must not share a hardware channel
        const char* mc = std::getenv("CUDA_DEVICE_MAX_CONNECTIONS");
        static bool warned = false;
        if (!warned && (!mc || std::atoi(mc) < 32)) {
            fprintf(stderr, "[liorf_b200] warning: CUDA_DEVICE_MAX_CONNECTIONS is %s; export CUDA_DEVICE_MAX_CONNECTIONS=32 before the first CUDA call when several "
                            "query batches are in flight per GPU (streams sharing a hardware channel can deadlock the cross-GPU flag waits)\n", mc ? mc : "unset (8)");
            warned = true;
        }
    }
    std::memset(&S.W, 0, sizeof(S.W));
    S.W.rank = rank; S.W.world = world; S.W.qmax = q_max; S.qmax = q_max; S.kcap = k_total_max;
    S.W.off_c = scsh_round((size_t)SCSH_MAX * SCSH_NPHASE * sizeof(unsigned));
    S.W.off_d = S.W.off_c + scsh_round((size_t)q_max * 24);
    S.off_keys = S.W.off_d + scsh_round((size_t)q_max * 36);
    S.win_bytes = S.off_keys + scsh_round((size_t)k_total_max * SC_RING * sizeof(float));
    CUDA_TRY(dev_alloc(S.win, S.win_bytes));
    unsigned char* win = S.win;
    CUDA_TRY(cudaMemset(win, 0, S.win_bytes));
    CUDA_TRY(dev_alloc(S.d_counter, 4 + SCSH_NPHASE * sizeof(unsigned long long) / sizeof(unsigned)));
    CUDA_TRY(cudaMemset(S.d_counter, 0, 4 * sizeof(unsigned) + SCSH_NPHASE * sizeof(unsigned long long)));
    S.d_nlist = reinterpret_cast<int*>(S.d_counter + 2);
    S.d_batch = S.d_counter + 1;
    S.W.wait_ns = reinterpret_cast<unsigned long long*>(S.d_counter + 4);
    S.W.base[rank] = win;
    if (ipc_handle_out) { cudaIpcMemHandle_t h; CUDA_TRY(cudaIpcGetMemHandle(&h, win)); static_assert(sizeof(h) == 64, "ipc handle"); std::memcpy(ipc_handle_out, &h, 64); }
    if (window_out) *window_out = win;
    return LIORF_OK;
}
/* nanoseconds this rank's kernels spent waiting for the peers' pushes, per phase (C, D, KEYS, unused), accumulated since the last call; batches = batch counter */
int liorf_sc_shard_wait_stats(liorf_ctx* c, unsigned long long wait_ns[4], unsigned* batches) {
    LIORF_NVTX;
    if (!c || !wait_ns) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    liorf_ctx::ScShard& S = c->shard;
    if (!S.d_counter) return LIORF_ERR_STATE;
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    CUDA_TRY(cudaMemcpy(wait_ns, S.W.wait_ns, SCSH_NPHASE * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    if (batches) CUDA_TRY(cudaMemcpy(batches, S.d_batch, sizeof(unsigned), cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemset(S.W.wait_ns, 0, SCSH_NPHASE * sizeof(unsigned long long)));
    return LIORF_OK;
}
int liorf_sc_shard_connect(liorf_ctx* c, const void* ipc_handles /*world x 64 B, nullable*/, void* const* window_ptrs /*world entries, nullable*/, const int* row_begin /*world + 1*/) {
    LIORF_NVTX;
    if (!c || (!ipc_handles && !window_ptrs) || !row_begin) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    liorf_ctx::ScShard& S = c->shard;
    if (!S.W.base[S.W.rank] || S.ready) return LIORF_ERR_STATE;
    if (row_begin[0] != 0) return LIORF_ERR_ARG;
    for (int g = 0; g <= S.W.world; ++g) { S.W.row_begin[g] = row_begin[g]; if (g > 0 && row_begin[g] < row_begin[g - 1]) return LIORF_ERR_ARG; }
    if (row_begin[S.W.world] < 1) return LIORF_ERR_ARG;                               // an empty DATABASE cannot be searched; an empty SHARD is fine
    if (S.kcap > 0 && row_begin[S.W.world] > S.kcap) return LIORF_ERR_ARG;            // the replicated index must hold every row
    // this rank's own rows must be the ones the context holds (a mismatch would make ranks disagree about who owns a candidate)
    if (c->sc_n != row_begin[S.W.rank + 1] - row_begin[S.W.rank]) return LIORF_ERR_STATE;
    for (int g = 0; g < S.W.world; ++g) {
        if (g != S.W.rank) {
            if (window_ptrs) S.W.base[g] = (unsigned char*)window_ptrs[g];               // same process: the peer context's pointer is directly usable
            else {
                cudaIpcMemHandle_t h; std::memcpy(&h, (const unsigned char*)ipc_handles + (size_t)64 * g, 64);
                CUDA_TRY(ipc_open(S.ipc[g], h));
                S.W.base[g] = S.ipc[g];
            }
            if (!S.W.base[g]) return LIORF_ERR_ARG;
        }
        S.W.keys_all[g] = S.kcap > 0 ? reinterpret_cast<float*>(S.W.base[g] + S.off_keys) : nullptr;     // every rank uses the same window layout
    }
    S.ready = true;
    return LIORF_OK;
}
/* Replicates the index: bit 0 = push the ring keys of this rank's rows into every rank's key array and raise the flags, bit 1 = wait for
 * every peer's keys (the next search rebuilds the operand image).  Collective: every rank calls it after the database was loaded or has
 * grown (liorf_sc_shard_sync_keys = both bits; the split form lets several ranks that share ONE device — tests — enqueue push before wait). */
int liorf_sc_shard_sync_keys_phases(liorf_ctx* c, int phases) {
    LIORF_NVTX;
    if (!c || !(phases & 3)) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    liorf_ctx::ScShard& S = c->shard;
    if (!S.ready || S.kcap < 1) return LIORF_ERR_STATE;
    if (c->sc_n != S.W.row_begin[S.W.rank + 1] - S.W.row_begin[S.W.rank]) return LIORF_ERR_STATE;
    if (phases & 1) {
        ++S.keys_gen; S.keys_pushed = true;
        const size_t words = (size_t)c->sc_n * SC_RING;
        const int blocks = (int)std::max<size_t>(1, std::min<size_t>(4 * c->num_sms, (words + 1023) / 1024));
        k_scsh_push_keys<<<blocks, 256, 0, c->stream>>>(S.W, c->sc_db->keys.p, c->sc_n, S.keys_gen, S.d_counter);
        CUDA_TRY(cudaGetLastError());
        c->launches += 1;
    }
    if (phases & 2) {
        if (!S.keys_pushed) return LIORF_ERR_STATE;
        k_scsh_wait_keys<<<1, 32, 0, c->stream>>>(S.W, S.keys_gen, c->d_err);
        CUDA_TRY(cudaGetLastError());
        c->ks_all.keys = S.W.keys_all[S.W.rank]; c->ks_all.n = S.W.row_begin[S.W.world]; c->ks_all.gen = S.keys_gen;
        c->launches += 1;
        return check_err(c);
    }
    return LIORF_OK;
}
int liorf_sc_shard_sync_keys(liorf_ctx* c) { return liorf_sc_shard_sync_keys_phases(c, 3); }
/* debugging aid: out[0] = batch counter, out[1] = raise counter, out[2] = owned-pair counter, out[3] = device error flag,
 * out[4 + 4 g + p] = flag of source rank g, phase p (C, D, KEYS, -) as it stands in THIS rank's window.  Synchronises the device. */
int liorf_sc_shard_debug_state(liorf_ctx* c, unsigned out[4 + 4 * 16]) {
    if (!c || !out) return LIORF_ERR_ARG;
    liorf_ctx::ScShard& S = c->shard;
    if (!S.d_counter || !S.W.base[S.W.rank]) return LIORF_ERR_STATE;
    CUDA_TRY(cudaSetDevice(c->P.device));
    CUDA_TRY(cudaDeviceSynchronize());
    unsigned cnt[4];
    CUDA_TRY(cudaMemcpy(cnt, S.d_counter, sizeof(cnt), cudaMemcpyDeviceToHost));
    out[0] = cnt[1]; out[1] = cnt[0]; out[2] = cnt[2];
    CUDA_TRY(cudaMemcpy(&out[3], c->d_err, sizeof(int), cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(out + 4, S.W.base[S.W.rank], (size_t)SCSH_MAX * SCSH_NPHASE * sizeof(unsigned), cudaMemcpyDeviceToHost));
    return LIORF_OK;
}
/* measurement only: 1 = this rank's consumer kernels do not wait for the peers' flags (a single rank of a G-rank search timed alone on one GPU
 * against windows that a complete earlier batch has filled; tools/profile_sc_shard.py) */
int liorf_sc_shard_debug_nowait(liorf_ctx* c, int on) {
    LIORF_NVTX;
    if (!c) return LIORF_ERR_ARG;
    c->shard.W.nowait = on != 0;
    c->shard.graph.reset();
    return LIORF_OK;
}

/* One query batch of the sharded search, enqueued on the context's stream (asynchronous; results on the device).  Every rank calls it
 * with the SAME queries in the same order.  phases: bit 0 = stage 1 of this rank's query slice (+ push C), bit 1 = collect + stage 2 of
 * the owned pairs (+ push D), bit 2 = decision. */
int liorf_sc_shard_query_phases_dev(liorf_ctx* c, const void* d_qdescs, int Q, int global_offset, void* d_loop_id, void* d_shift, void* d_dist, void* d_cand, int phases) {
    LIORF_NVTX;
    if (!c || !d_qdescs || Q < 1 || !d_loop_id || !d_shift || !d_dist || !(phases & 7)) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    liorf_ctx::ScShard& S = c->shard;
    if (!S.ready || Q > S.qmax) return LIORF_ERR_STATE;
    // ownership must be the one every rank agreed on at connect time (a database that has grown needs a new connect + key sync)
    if (global_offset != S.W.row_begin[S.W.rank] || c->sc_n != S.W.row_begin[S.W.rank + 1] - S.W.row_begin[S.W.rank]) return LIORF_ERR_STATE;
    int rc;
    const double* qd = (const double*)d_qdescs;
    int* cand = d_cand ? (int*)d_cand : c->sc_q_i.p;
    if (S.W.world == 1) {                        // one rank: nothing to exchange → the plain search (the same kernels)
        if (phases != 7) return LIORF_ERR_ARG;
        if (c->sc_n < 1) return LIORF_ERR_STATE;
        if ((rc = sc_reserve_query(c, Q))) return rc;
        if (!d_cand) cand = c->sc_q_i.p;
        return sc_query_local_dev(c, qd, Q, global_offset, cand, (int*)d_loop_id, (int*)d_shift, (double*)d_dist);
    }
    liorf_ctx::KeySet& ks = c->ks_all;
    if (!ks.keys || ks.n != S.W.row_begin[S.W.world]) return LIORF_ERR_STATE;       // liorf_sc_shard_sync_keys (or a borrow from a synced context) first
    const int q0 = (int)((long long)Q * S.W.rank / S.W.world), q1 = (int)((long long)Q * (S.W.rank + 1) / S.W.world), Qs = q1 - q0;
    if ((rc = c->sc_qkeys.reserve((size_t)std::max(Qs, 1) * SC_RING)) || (rc = sc_reserve_query(c, Q)) || (rc = S.list.reserve((size_t)3 * Q))) return rc;
    if (!d_cand) cand = c->sc_q_i.p;
    ShardPush P; std::memset(&P, 0, sizeof(P));
    P.enabled = 1; P.q0 = q0; P.W = S.W; P.counter = S.d_counter; P.batch_p = S.d_batch;
    if (phases & 1) {        // ring keys of this rank's query slice (first block bumps the batch number) → exact GLOBAL top-3 → every window
        if (((uintptr_t)qd & 15) == 0) k_sc_ringkeys_batch<<<(std::max(Qs, 1) + SCK_WARPS - 1) / SCK_WARPS, 32 * SCK_WARPS, 0, c->stream>>>(qd + (size_t)q0 * SC_DESC, Qs, c->sc_qkeys.p, S.d_batch);
        else k_sc_keys_batch<<<std::max(Qs, 1), 64, 0, c->stream>>>(qd + (size_t)q0 * SC_DESC, Qs, c->sc_qkeys.p, nullptr, nullptr, S.d_batch);
        c->launches += 1;
        if (Qs > 0 && sc_want_tensor(c, Qs, ks.n)) { if ((rc = sc_knn_tensor(c, ks, ks.n, c->sc_qkeys.p, Qs, 0, nullptr, nullptr, &P))) return rc; }
        else {
            if (Qs > 0 && (rc = sc_knn_brute(c, ks.keys, ks.n, c->sc_qkeys.p, Qs, 0, c->sc_q_d.p, c->sc_q_i.p))) return rc;
            k_scsh_push_c<<<std::max(1, std::min(64, (3 * Qs + 255) / 256)), 256, 0, c->stream>>>(S.W, c->sc_q_d.p, c->sc_q_i.p, q0, Qs, S.d_batch, S.d_counter);
            c->launches += 1;
        }
    }
    if (phases & 2) {        // every slice has arrived → local copy + the pairs this rank owns → distanceBtnScanContext on exactly those, pushed by the warps that compute them
        k_scsh_wait_phase<<<1, 32, 0, c->stream>>>(S.W, SCSH_C, S.d_batch, c->d_err);
        k_scsh_collect<<<(Q + 127) / 128, 128, 0, c->stream>>>(S.W, S.d_batch, Q, c->sc_q_d.p, cand, c->d_err, global_offset, c->sc_n, S.list.p, S.d_nlist);
        c->launches += 2;
        if ((rc = sc_distance_launch(c, qd, cand, 3 * Q, global_offset, nullptr, nullptr, S.list.p, S.d_nlist, &P))) return rc;
    }
    if (phases & 4) {        // decision (+ re-arms the owned-pair counter)
        k_scsh_wait_phase<<<1, 32, 0, c->stream>>>(S.W, SCSH_D, S.d_batch, c->d_err);
        k_scsh_decide<<<(Q + 127) / 128, 128, 0, c->stream>>>(S.W, S.d_batch, cand, Q, (int*)d_loop_id, (int*)d_shift, (double*)d_dist, c->d_err, S.d_nlist);
        c->launches += 2;
    }
    CUDA_TRY(cudaGetLastError());
    return LIORF_OK;
}
/* One query batch of the sharded search, enqueued on the context's stream (asynchronous; results on the device).  Every rank calls it
 * with the SAME queries in the same order. */
int liorf_sc_shard_query_dev(liorf_ctx* c, const void* d_qdescs, int Q, int global_offset, void* d_loop_id, void* d_shift, void* d_dist, void* d_cand) {
    LIORF_NVTX;
    if (!c) return LIORF_ERR_ARG;
    liorf_ctx::ScShard& S = c->shard;
    // A batch is ~9 small kernels: replayed from a CUDA graph once the same request has been seen twice, so that the host's launch rate does
    // not bound the queries/s.  The signature holds everything a captured kernel argument can depend on: the caller's buffers and sizes, the
    // database extent and key generation, the search path, and every internal buffer (DevBuf::reserve may reallocate any of them).
    const bool can_graph = c->use_graphs && !c->prof.enabled && S.ready;
    if (!can_graph) return liorf_sc_shard_query_phases_dev(c, d_qdescs, Q, global_offset, d_loop_id, d_shift, d_dist, d_cand, 7);
    auto make_sig = [&](const void** sig) {
        const liorf_ctx::KeySet& ks = S.W.world == 1 ? c->ks_local : c->ks_all;
        const void* v[40] = {d_qdescs, (const void*)(size_t)Q, (const void*)(size_t)global_offset, d_loop_id, d_shift, d_dist, d_cand, (const void*)(size_t)c->sc_n,
                             (const void*)(size_t)ks.n, (const void*)(size_t)ks.gen, (const void*)(size_t)ks.img_n, (const void*)(size_t)ks.img_gen, ks.keys, ks.bimg.p, ks.center,
                             (const void*)(size_t)c->sc_path, (const void*)(size_t)S.W.nowait,
                             c->sc_db->desc.p, c->sc_db->sk.p, c->sc_db->cn.p, c->sc_db->keys.p, c->sc_qkeys.p, c->sc_q_d.p, c->sc_q_i.p, c->sc_pair_d.p, c->sc_pair_s.p, c->sc_part_d.p, c->sc_part_i.p,
                             S.list.p, c->sct_aimg.p, c->sct_qnorm.p, c->sct_cmin.p, c->sct_cmin32.p, c->sct_part.p, c->sct_cand.p, c->sct_cnt.p, c->sct_over_cnt, nullptr, nullptr, nullptr};
        std::memcpy(sig, v, sizeof(v));
    };
    const void* sig[40];
    make_sig(sig);
    if (S.graph && std::memcmp(sig, S.gsig, sizeof(sig)) == 0) {
        CUDA_TRY(cudaSetDevice(c->P.device));
        CUDA_TRY(cudaGraphLaunch(S.graph, c->stream));
        c->launches += 11;
        return LIORF_OK;
    }
    if (std::memcmp(sig, S.last_sig, sizeof(sig)) == 0) {        // second identical request: every buffer is sized and the operand image is current → capture
        CUDA_TRY(cudaSetDevice(c->P.device));
        S.graph.reset();
        Graph g;
        const long long launches0 = c->launches;
        CUDA_TRY(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
        const int rc = liorf_sc_shard_query_phases_dev(c, d_qdescs, Q, global_offset, d_loop_id, d_shift, d_dist, d_cand, 7);
        const cudaError_t e = end_capture(g, c->stream);
        c->launches = launches0;
        if (rc || e != cudaSuccess) { (void)cudaGetLastError(); return rc ? rc : LIORF_ERR_CUDA; }
        make_sig(sig);
        if (std::memcmp(sig, S.last_sig, sizeof(sig)) != 0) {     // something was (re)allocated or rebuilt during the capture after all: do not keep it
            std::memset(S.last_sig, 0, sizeof(S.last_sig));
            return liorf_sc_shard_query_phases_dev(c, d_qdescs, Q, global_offset, d_loop_id, d_shift, d_dist, d_cand, 7);
        }
        CUDA_TRY(graph_instantiate(S.graph, g));
        std::memcpy(S.gsig, sig, sizeof(sig));
        CUDA_TRY(cudaGraphLaunch(S.graph, c->stream));
        c->launches += 11;
        return LIORF_OK;
    }
    const int rc = liorf_sc_shard_query_phases_dev(c, d_qdescs, Q, global_offset, d_loop_id, d_shift, d_dist, d_cand, 7);
    make_sig(S.last_sig);                                         // as of AFTER the call: buffers sized, image built
    return rc;
}

/* The sharded batch from HOST buffers (the reference-facing form: detectLoopClosureID's inputs and answers live in host memory):
 * H2D of the Q query descriptors, liorf_sc_shard_query_dev, D2H of the answers — all asynchronous on the context's stream; the host
 * buffers (pinned for real asynchrony) must stay valid and the results are defined after liorf_sync.  cand3 nullable. */
int liorf_sc_shard_query_async(liorf_ctx* c, const double* qdescs, int Q, int global_offset, int* loop_id, int* shift, double* dist, int* cand3) {
    LIORF_NVTX;
    if (!c || !qdescs || Q < 1 || !loop_id || !shift || !dist) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    int rc;
    if ((rc = c->sc_qdesc.reserve((size_t)Q * SC_DESC)) || (rc = sc_reserve_query(c, Q))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->sc_qdesc.p, qdescs, (size_t)Q * SC_DESC * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    if ((rc = liorf_sc_shard_query_dev(c, c->sc_qdesc.p, Q, global_offset, c->sc_res_i.p, c->sc_res_i.p + Q, c->sc_res_d.p, c->sc_q_i.p))) return rc;
    CUDA_TRY(cudaMemcpyAsync(loop_id, c->sc_res_i.p, (size_t)Q * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(shift, c->sc_res_i.p + Q, (size_t)Q * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(dist, c->sc_res_d.p, (size_t)Q * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    if (cand3) CUDA_TRY(cudaMemcpyAsync(cand3, c->sc_q_i.p, (size_t)3 * Q * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    return LIORF_OK;
}

// yawDiffRad of detectLoopClosureID from the decided column shift: deg2rad(float) of the shift in degrees (:17-20, :339)
static float sc_yaw_rad(int nn_align) { return (float)((float)(nn_align * (360.0 / 60.0)) * M_PI / 180.0); }

int liorf_sc_detect_loop_closure_id(liorf_ctx* c, int* loop_id, float* yaw_diff_rad, double* min_dist, int* cand3) {
    LIORF_NVTX;
    if (!c || !loop_id || !yaw_diff_rad) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    *loop_id = -1; *yaw_diff_rad = 0.f;
    if (c->sc_n < SC_EXCLUDE_RECENT + 1) return LIORF_OK;                       // :263-267
    if (c->sc_counter % SC_TREE_PERIOD == 0) c->sc_tree_n = c->sc_n - SC_EXCLUDE_RECENT;   // :270-281 (tree snapshot = keys[0 : n-30])
    c->sc_counter = c->sc_counter + 1;
    int rc;
    if ((rc = sc_reserve_query(c, 1))) return rc;
    const size_t qe = (size_t)c->sc_n - 1;                                       // query = last entry (:257-258)
    if ((rc = sc_knn(c, local_keys(c), c->sc_tree_n, c->sc_db->keys.p + qe * SC_RING, 1, 0, c->sc_q_d.p, c->sc_q_i.p))) return rc;
    // result slots are zero-initialised in the reference (:289-290): an unfilled slot means candidate 0
    CUDA_TRY(cudaMemcpyAsync(c->h_mail.p + 700, c->sc_q_i.p, 3 * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    int cand[3]; for (int j = 0; j < 3; ++j) { cand[j] = c->h_mail.p[700 + j]; if (cand[j] == 0x7fffffff) cand[j] = 0; c->h_mail.p[704 + j] = cand[j]; }
    CUDA_TRY(cudaMemcpyAsync(c->sc_q_i.p, c->h_mail.p + 704, 3 * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    k_sc_distance<<<1, SCD_WARPS * 32, 0, c->stream>>>(c->sc_db->desc.p + qe * SC_DESC, c->sc_db->sk.p + qe * SC_SECTOR, c->sc_db->cn.p + qe * SC_SECTOR, c->sc_q_i.p, 3, 3,
                                                       c->sc_db->desc.p, c->sc_db->sk.p, c->sc_db->cn.p, 0, c->sc_n, c->sc_pair_d.p, c->sc_pair_s.p);
    k_sc_decide<<<1, 128, 0, c->stream>>>(c->sc_pair_d.p, c->sc_pair_s.p, c->sc_q_i.p, 1, c->sc_res_i.p, c->sc_res_i.p + 1, c->sc_res_d.p);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(c->h_mail.p + 710, c->sc_res_i.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(c->h_mail.p + 720, c->sc_res_d.p, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    if ((rc = check_err(c))) return rc;
    *loop_id = c->h_mail.p[710];
    const int nn_align = c->h_mail.p[711];
    double md; std::memcpy(&md, c->h_mail.p + 720, sizeof(double));
    if (min_dist) *min_dist = md;
    if (cand3) { cand3[0] = cand[0]; cand3[1] = cand[1]; cand3[2] = cand[2]; }
    *yaw_diff_rad = sc_yaw_rad(nn_align);
    return LIORF_OK;
}

/* detectLoopClosureID for Q calls at once (header): query q is row n_db[q] - 1, searched over keys [0, n_tree[q]).  Queries past the
 * early-out are gathered into contiguous query buffers; stage 1 runs with per-query key limits, stage 2 and the decision are the batch
 * search's kernels.  Device layout of scdb_io (ints, Qd gathered queries): dist f64[Qd] | loop_id[Qd] | shift[Qd] | cand[3 Qd] | n_db[Qd] |
 * n_tree[Qd] — the first 7 Qd ints come back in one copy, the last 2 Qd go up in one. */
int liorf_sc_detect_loop_closure_id_batch(liorf_ctx* c, const int* n_db, const int* n_tree, int Q, int* loop_id, float* yaw_diff_rad, double* min_dist, int* cand3) {
    LIORF_NVTX;
    if (!c || Q < 0 || (Q > 0 && (!n_db || !n_tree || !loop_id || !yaw_diff_rad))) return LIORF_ERR_ARG;
    int Qd = 0, max_tree = 0, min_tree = 0x7fffffff;
    for (int q = 0; q < Q; ++q) {
        if (n_db[q] < 1 || n_db[q] > c->sc_n) return LIORF_ERR_ARG;
        if (n_db[q] < SC_EXCLUDE_RECENT + 1) continue;                          // :263-267
        if (n_tree[q] < 1 || n_tree[q] > n_db[q] - SC_EXCLUDE_RECENT) return LIORF_ERR_ARG;
        ++Qd; max_tree = std::max(max_tree, n_tree[q]); min_tree = std::min(min_tree, n_tree[q]);
    }
    if (Q == 0) return LIORF_OK;
    CUDA_TRY(cudaSetDevice(c->P.device));
    int rc;
    if (Qd > 0) {
        const size_t io_ints = (size_t)9 * Qd;
        if (io_ints > c->h_scdb.cap) {
            if (c->h_scdb.p) CUDA_TRY(cudaStreamSynchronize(c->stream));
            if ((rc = c->h_scdb.reserve(std::max<size_t>(io_ints, 1 << 16)))) return rc;
        }
        if ((rc = c->scdb_io.reserve(io_ints)) || (rc = c->sc_qdesc.reserve((size_t)Qd * SC_DESC)) || (rc = c->sc_qkeys.reserve((size_t)Qd * SC_RING)) ||
            (rc = sc_reserve_query(c, Qd))) return rc;
        int* H = c->h_scdb.p;
        for (int q = 0, k = 0; q < Q; ++q)
            if (n_db[q] >= SC_EXCLUDE_RECENT + 1) { H[7 * Qd + k] = n_db[q]; H[8 * Qd + k] = n_tree[q]; ++k; }
        int* D = c->scdb_io.p;
        double* d_dist = reinterpret_cast<double*>(D);
        int *d_loop = D + 2 * Qd, *d_shift = D + 3 * Qd, *d_cand = D + 4 * Qd, *d_rows = D + 7 * Qd, *d_lim = D + 8 * Qd;
        CUDA_TRY(cudaMemcpyAsync(d_rows, H + 7 * Qd, (size_t)2 * Qd * sizeof(int), cudaMemcpyHostToDevice, c->stream));
        k_sc_gather_queries<<<Qd, 128, 0, c->stream>>>(c->sc_db->desc.p, c->sc_db->keys.p, d_rows, Qd, c->sc_qdesc.p, c->sc_qkeys.p);
        CUDA_TRY(cudaGetLastError());
        c->launches += 1;
        // stage 1 on the path the batch search would take for Qd queries against this database; the CUDA-core kernel needs to look no
        // further than the largest limit, the tensor-core filter keeps the database's operand image
        if (sc_want_tensor(c, Qd, c->sc_n)) rc = sc_knn_tensor(c, local_keys(c), c->sc_n, c->sc_qkeys.p, Qd, 0, c->sc_q_d.p, d_cand, nullptr, d_lim);
        else rc = sc_knn_brute(c, c->sc_db->keys.p, max_tree, c->sc_qkeys.p, Qd, 0, c->sc_q_d.p, d_cand, d_lim);
        if (rc) return rc;
        if (min_tree < SC_NUM_CAND) {
            k_sc_cand_unfilled_to_zero<<<(3 * Qd + 127) / 128, 128, 0, c->stream>>>(d_cand, 3 * Qd);
            CUDA_TRY(cudaGetLastError());
            c->launches += 1;
        }
        if ((rc = sc_distance_launch(c, c->sc_qdesc.p, d_cand, 3 * Qd, 0, c->sc_pair_d.p, c->sc_pair_s.p))) return rc;
        if ((rc = liorf_sc_decide_dev(c, c->sc_pair_d.p, c->sc_pair_s.p, d_cand, Qd, d_loop, d_shift, d_dist))) return rc;
        CUDA_TRY(cudaMemcpyAsync(H, D, (size_t)7 * Qd * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        if ((rc = check_err(c))) return rc;
    }
    const int* H = c->h_scdb.p;
    for (int q = 0, k = 0; q < Q; ++q) {
        loop_id[q] = -1; yaw_diff_rad[q] = 0.f;
        if (n_db[q] < SC_EXCLUDE_RECENT + 1) continue;
        loop_id[q] = H[2 * Qd + k];
        yaw_diff_rad[q] = sc_yaw_rad(H[3 * Qd + k]);
        if (min_dist) std::memcpy(min_dist + q, H + 2 * (size_t)k, sizeof(double));
        if (cand3) for (int j = 0; j < 3; ++j) cand3[3 * (size_t)q + j] = H[4 * Qd + 3 * k + j];
        ++k;
    }
    return LIORF_OK;
}


// ------------------------------------------------------------------------------------------------ loop-closure ICP
// clouds of loopFindNearKeyframes (:821-844) as performSCLoopClosure calls it (:652-653): every selected keyframe cloud is
// transformed by the pose of keyframe `loop_index` (the reference passes base_key = 0), concatenated, VoxelGrid(icp leaf).
// loopFindNearKeyframes' selection (:826-835): keyframes key-search_num .. key+search_num that exist, in order; appends to sel with
// destination offsets continuing from `total`.  sel == nullptr only counts the points.
static void icp_select(const liorf_ctx* c, int key, int search_num, int loop_index, std::vector<KfSel>* sel, long long& total) {
    const int n_kf = (int)c->kfs.size();
    for (int i = -search_num; i <= search_num; ++i) {
        const int kn = key + i;
        if (kn < 0 || kn >= n_kf) continue;
        const Keyframe& k = c->kfs[kn];
        if (sel) {
            const Keyframe& pk = c->kfs[loop_index != -1 ? loop_index : kn];
            KfSel s; s.src_off = (int)k.off; s.count = k.count; s.dst_off = (int)total; s.pad = 0;
            host_get_transformation(pk.pose[3], pk.pose[4], pk.pose[5], pk.pose[0], pk.pose[1], pk.pose[2], s.t);
            sel->push_back(s);
        }
        total += k.count;
    }
}

static int icp_build_cloud(liorf_ctx* c, int key, int search_num, int loop_index, float leaf, DevBuf<float4>& out, int* n_out) {
    int rc;
    std::vector<KfSel> sel; long long total = 0;
    icp_select(c, key, search_num, loop_index, &sel, total);
    *n_out = 0;
    if (sel.empty() || total == 0) return LIORF_OK;
    if (total > 0x7fffffffLL) return LIORF_ERR_ARG;
    const int tot = (int)total, ns = (int)sel.size();
    if ((rc = c->icp_sel.reserve(ns)) || (rc = c->icp_raw.reserve(tot)) || (rc = out.reserve(tot))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->icp_sel.p, sel.data(), (size_t)ns * sizeof(KfSel), cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));                      // `sel` is pageable host memory going out of scope
    k_transform_concat<<<(tot + 255) / 256, 256, 0, c->stream>>>(c->kf_points.p, c->icp_sel.p, ns, tot, c->icp_raw.p);
    if ((rc = voxel_grid_device(c->icp_raw.p, Count::of_host(tot), leaf, out.p, c->d_counts + C_HOOK_NSEL, nullptr, nullptr, c->vg, c->stream))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->h_mail.p + 900, c->d_counts + C_HOOK_NSEL, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    *n_out = c->h_mail.p[900];
    c->launches += 10;
    return LIORF_OK;
}

// the result fields of a pair that ran, from the loop state and getFitnessScore's two sums (shared by the single and the batched call)
static void icp_fill_result(const IcpState& hs, const double* fit_sums, liorf_icp_result* out) {
    out->ran = 1;
    out->iterations = hs.iterations;
    out->converged = hs.converged ? 1 : 0; out->convergence_state = (int)hs.cc.state;
    std::memcpy(out->transform, hs.final_T, sizeof(hs.final_T));
    out->fitness = fit_sums[1] > 0 ? (float)(fit_sums[0] / fit_sums[1]) : 3.4028235e38f;
    float t12[12]; for (int r = 0; r < 3; ++r) for (int k = 0; k < 4; ++k) t12[4 * r + k] = hs.final_T[4 * r + k];
    liorf_host::get_translation_and_euler(t12, out->pose6[3], out->pose6[4], out->pose6[5], out->pose6[0], out->pose6[1], out->pose6[2]);   // :693
}
constexpr int ICP_CHUNK = 8;                         // iterations enqueued between two read-backs of the loop state
static IcpState icp_initial_state(int max_iters) {
    IcpState hs; std::memset(&hs, 0, sizeof(hs));
    hs.cc = liorf_host::IcpConvergence(); hs.cc.max_iterations = max_iters;
    for (int i = 0; i < 4; ++i) hs.inc[5 * i] = hs.final_T[5 * i] = 1.f;
    return hs;
}

int liorf_loop_closure_icp(liorf_ctx* c, int loop_key_cur, int loop_key_pre, int history_search_num, int loop_index, float icp_leaf, float max_corr_dist,
                           int max_iters, liorf_icp_result* out) {
    LIORF_NVTX;
    if (!c || !out || history_search_num < 0 || max_iters < 1 || !(icp_leaf > 0.f) || !(max_corr_dist > 0.f)) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    std::memset(out, 0, sizeof(*out));
    for (int i = 0; i < 4; ++i) out->transform[5 * i] = 1.f;
    const int n_kf = (int)c->kfs.size();
    if (loop_key_cur < 0 || loop_key_cur >= n_kf || loop_key_pre < 0 || loop_key_pre >= n_kf || loop_index < -1 || loop_index >= n_kf) return LIORF_ERR_ARG;
    int rc;
    if ((rc = join_map(c))) return rc;
    int n_src = 0, n_tgt = 0;
    if ((rc = icp_build_cloud(c, loop_key_cur, 0, loop_index, icp_leaf, c->icp_src0, &n_src))) return rc;                 // cureKeyframeCloud  (:652)
    if ((rc = icp_build_cloud(c, loop_key_pre, history_search_num, loop_index, icp_leaf, c->icp_tgt, &n_tgt))) return rc;   // prevKeyframeCloud  (:653)
    out->n_source = n_src; out->n_target = n_tgt;
    if (n_src < 300 || n_tgt < 1000) return check_err(c);           // :655-656
    out->ran = 1;
    if (!c->icp_out) { CUDA_TRY(dev_alloc(c->icp_out, ICP_NSUM)); c->icp_counter = c->d_misc + 14; }
    int blocks = (n_src + ICP_BLOCK - 1) / ICP_BLOCK; if (blocks > 4 * c->num_sms) blocks = 4 * c->num_sms;
    if ((rc = c->icp_partial.reserve((size_t)blocks * ICP_NSUM)) || (rc = c->icp_src.reserve(n_src))) return rc;
    if ((rc = build_map_grid(c->icp_tgt.p, Count::of_host(n_tgt), c->icp_grid, c->stream))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->icp_src.p, c->icp_src0.p, (size_t)n_src * sizeof(float4), cudaMemcpyDeviceToDevice, c->stream));
    const int r_max = (int)std::ceil(max_corr_dist) + 1;
    const float max_d2 = max_corr_dist * max_corr_dist;
    // the loop runs on the device (csrc/icp.cuh): iterations are enqueued in chunks and the state is read back once per chunk
    if (!c->icp_state) CUDA_TRY(dev_alloc(c->icp_state, 1));
    IcpState hs = icp_initial_state(max_iters);
    CUDA_TRY(cudaMemcpyAsync(c->icp_state, &hs, sizeof(hs), cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));                       // hs is pageable: the copy must have left it before it is reused below
    int enq = 0;
    while (!hs.done && enq < max_iters) {
        const int todo = std::min(ICP_CHUNK, max_iters - enq);
        for (int k = 0; k < todo; ++k)
            k_icp_iteration<<<blocks, ICP_BLOCK, 0, c->stream>>>(c->icp_src.p, n_src, c->icp_state, c->icp_grid.cell_start.p, c->icp_grid.sorted.p, c->icp_grid.dims, r_max, max_d2,
                                                               c->icp_partial.p, c->icp_counter, c->icp_out, nullptr, nullptr);
        enq += todo; c->launches += todo;
        CUDA_TRY(cudaMemcpyAsync(&hs, c->icp_state, sizeof(hs), cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(cudaStreamSynchronize(c->stream));
    }
    double* h_sums = reinterpret_cast<double*>(c->h_mail.p + 3000);   // 8-byte aligned slot of the pinned mailbox
    // getFitnessScore(): the original source under the final transformation, no range limit
    {
        IcpT Tf; std::memcpy(Tf.t, hs.final_T, 12 * sizeof(float));
        const int rfit = 64;
        k_icp_fitness<<<blocks, ICP_BLOCK, 0, c->stream>>>(c->icp_src0.p, n_src, Tf, c->icp_grid.cell_start.p, c->icp_grid.sorted.p, c->icp_grid.dims, rfit, c->icp_partial.p,
                                                         c->icp_counter, c->icp_out);
        CUDA_TRY(cudaMemcpyAsync(h_sums, c->icp_out, 2 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(cudaStreamSynchronize(c->stream));
        ++c->launches;
    }
    icp_fill_result(hs, h_sums, out);
    return check_err(c);
}
/* test hook: the two clouds of the last liorf_loop_closure_icp (cureKeyframeCloud / prevKeyframeCloud after the ICP VoxelGrid) */
int liorf_icp_get_clouds(liorf_ctx* c, liorf_point* source, int cap_source, liorf_point* target, int cap_target) {
    LIORF_NVTX;
    if (!c) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    if (source && cap_source > 0) CUDA_TRY(cudaMemcpy(source, c->icp_src0.p, (size_t)cap_source * sizeof(float4), cudaMemcpyDeviceToHost));
    if (target && cap_target > 0) CUDA_TRY(cudaMemcpy(target, c->icp_tgt.p, (size_t)cap_target * sizeof(float4), cudaMemcpyDeviceToHost));
    return LIORF_OK;
}

// ------------------------------------------------------------------------------------------------ batched loop-closure ICP
// liorf_loop_closure_icp for many pairs (icp_batch.cuh).  Pairs run in waves bounded by ICPB_WAVE_BYTES of work buffers; a wave costs
// one host synchronisation after its clouds are built (voxel counts per cloud), one per chunk of ICP_CHUNK iterations, one for the
// fitness sums, and the batch one error check — however many pairs the wave holds.
constexpr size_t ICPB_WAVE_BYTES = LIORF_ICP_BATCH_WAVE_BYTES;
constexpr size_t ICPB_BYTES_PER_POINT = 96;          // raw + voxel + working copy + cell-sorted copy (16 B each), sort keys / values / heads
constexpr size_t ICPB_GRID_BYTES = (size_t)256 * 256 * 32 * 2 * sizeof(unsigned);      // per pair: cell counts + cell starts
constexpr int ICPB_MAX_PAIRS = 256;                  // 512 clouds per wave; 2^29 grid cells

struct IcpbPair { int cur, pre, li; long long raw_src, raw_tgt; };

static int icpb_stage(liorf_ctx* c, size_t bytes) {   // pinned staging (grows between waves, when the stream is idle)
    HostBuf<unsigned char>& h = c->icpb.h_stage;
    if (bytes <= h.cap) return LIORF_OK;
    if (h.p) CUDA_TRY(cudaStreamSynchronize(c->stream));
    return h.reserve(std::max<size_t>(bytes, 1 << 20));
}

// one wave: pairs P[0 .. W).  *split = 1 (nothing written to out) when the wave's VoxelGrid keys need more than 32 bits: the caller halves it.
static int icpb_wave(liorf_ctx* c, const IcpbPair* P, int W, liorf_icp_result* const* out, int history_search_num, float leaf, float max_corr_dist,
                     int max_iters, int* split) {
    liorf_ctx::IcpBatch& B = c->icpb;
    cudaStream_t s = c->stream;
    int rc;
    *split = 0;
    // ---- selections of all 2 W clouds (cloud 2 j = pair j's source, 2 j + 1 its target), one tile table over them ----
    const int S = 2 * W;
    std::vector<KfSel> sel; std::vector<int> seg_n(S), seg_first(S); std::vector<VgSegTile> tiles;
    long long total = 0;
    for (int j = 0; j < W; ++j)
        for (int side = 0; side < 2; ++side) {
            const int sg = 2 * j + side;
            const long long t0 = total;
            if (side == 0) icp_select(c, P[j].cur, 0, P[j].li, &sel, total);                    // cureKeyframeCloud  (:652)
            else icp_select(c, P[j].pre, history_search_num, P[j].li, &sel, total);            // prevKeyframeCloud  (:653)
            seg_first[sg] = (int)t0; seg_n[sg] = (int)(total - t0);
            for (long long b = t0; b < total; b += VGSEG_TILE) tiles.push_back(VgSegTile{sg, (int)b, (int)std::min<long long>(b + VGSEG_TILE, total), 0});
        }
    const int tot = (int)total, ns = (int)sel.size(), nt = (int)tiles.size();
    // pinned staging: [up: sel | tiles | seg_n | seg_first | pair table | act (2 W) | states]  [down: seg_vox | flags | states | fitness sums]
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
    const size_t o_sel = take((size_t)ns * sizeof(KfSel)), o_tiles = take((size_t)nt * sizeof(VgSegTile)), o_segn = take((size_t)2 * S * sizeof(int));
    const size_t o_pd = take((size_t)W * sizeof(IcpPairDesc)), o_act = take((size_t)2 * W * sizeof(int2)), o_st = take((size_t)W * sizeof(IcpState));
    const size_t o_vox = take((size_t)2 * S * sizeof(int) + 2 * sizeof(int)), o_stb = take((size_t)W * sizeof(IcpState)), o_fit = take((size_t)2 * W * sizeof(double));
    if ((rc = icpb_stage(c, off))) return rc;
    unsigned char* H = B.h_stage.p;
    int* h_vox = reinterpret_cast<int*>(H + o_vox);           // [2 S] (first voxel, count) per cloud, then the two flags
    if (tot > 0) {
        std::memcpy(H + o_sel, sel.data(), (size_t)ns * sizeof(KfSel));
        std::memcpy(H + o_tiles, tiles.data(), (size_t)nt * sizeof(VgSegTile));
        std::memcpy(H + o_segn, seg_n.data(), (size_t)S * sizeof(int)); std::memcpy(H + o_segn + (size_t)S * sizeof(int), seg_first.data(), (size_t)S * sizeof(int));
        if ((rc = B.sel.reserve(ns)) || (rc = B.tiles.reserve(nt)) || (rc = B.seg_n.reserve((size_t)2 * S)) || (rc = B.seg_vox.reserve((size_t)2 * S)) ||
            (rc = B.mm.reserve((size_t)6 * S)) || (rc = B.metas.reserve(S)) || (rc = B.seg_base.reserve((size_t)S + 1)) || (rc = B.raw.reserve(tot)) ||
            (rc = B.keys.reserve(tot)) || (rc = B.seg_start.reserve((size_t)tot + 1)) || (rc = B.vox.reserve(tot))) return rc;
        CUDA_TRY(cudaMemcpyAsync(B.sel.p, H + o_sel, (size_t)ns * sizeof(KfSel), cudaMemcpyHostToDevice, s));
        CUDA_TRY(cudaMemcpyAsync(B.tiles.p, H + o_tiles, (size_t)nt * sizeof(VgSegTile), cudaMemcpyHostToDevice, s));
        CUDA_TRY(cudaMemcpyAsync(B.seg_n.p, H + o_segn, (size_t)2 * S * sizeof(int), cudaMemcpyHostToDevice, s));
        CUDA_TRY(cudaMemsetAsync(B.mm.p, 0xff, (size_t)3 * S * sizeof(unsigned), s));
        CUDA_TRY(cudaMemsetAsync(B.mm.p + 3 * S, 0, (size_t)3 * S * sizeof(unsigned), s));
        // ---- the clouds: one transform + concat, then the segmented VoxelGrid (voxelgrid.cuh) ----
        k_transform_concat<<<(tot + 255) / 256, 256, 0, s>>>(c->kf_points.p, B.sel.p, ns, tot, B.raw.p);
        k_vgseg_bounds<<<nt, 256, 0, s>>>(B.raw.p, B.tiles.p, B.mm.p, B.mm.p + 3 * S);
        k_vgseg_meta<<<1, 1024, 0, s>>>(B.seg_n.p, S, B.mm.p, B.mm.p + 3 * S, leaf, B.metas.p, B.seg_base.p, B.d_flags + 1);
        k_vgseg_keys<<<nt, 256, 0, s>>>(B.raw.p, B.tiles.p, B.seg_n.p + S, B.metas.p, B.seg_base.p, B.keys.p);
        unsigned* sorted_idx = nullptr;
        const Count cnt = Count::of_host(tot);
        if ((rc = radix_sort_pairs_iota(B.keys.p, cnt, B.sort, &sorted_idx, s))) return rc;
        if ((rc = launch_scan(cnt, VgHeadLoad{B.keys.p}, VgHeadStore{B.seg_start.p, cnt}, B.scan, (unsigned*)B.d_flags.get(), s))) return rc;
        k_vg_centroid<<<(tot + 127) / 128, 128, 0, s>>>(B.raw.p, sorted_idx, B.seg_start.p, (const unsigned*)B.d_flags.get(), B.vox.p, nullptr, B.keys.p, nullptr);
        k_vgseg_out<<<(S + 255) / 256, 256, 0, s>>>(B.keys.p, B.seg_start.p, (const unsigned*)B.d_flags.get(), B.seg_base.p, S, B.seg_vox.p);
        CUDA_TRY(cudaGetLastError());
        c->launches += 16;
        CUDA_TRY(cudaMemcpyAsync(h_vox, B.seg_vox.p, (size_t)2 * S * sizeof(int), cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaMemcpyAsync(h_vox + 2 * S, B.d_flags, 2 * sizeof(int), cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaStreamSynchronize(s));                                    // sync 1: voxel counts of every cloud
        if (h_vox[2 * S + 1] && W > 1) { *split = 1; return LIORF_OK; }
        if (h_vox[2 * S + 1]) {
            // one pair whose key ranges sum past 2^32 (a cloud near PCL's guard has a range up to ~2^32 by itself): the segmented keys
            // wrapped, so its two clouds are filtered one at a time from the same transformed points, as the single-pair call filters them
            int at = 0;
            for (int sg = 0; sg < S; ++sg) {
                if ((rc = voxel_grid_device(B.raw.p + seg_first[sg], Count::of_host(seg_n[sg]), leaf, B.vox.p + at, c->d_counts + C_HOOK_NSEL, nullptr, nullptr,
                                            c->vg, s))) return rc;
                CUDA_TRY(cudaMemcpyAsync(h_vox + 2 * sg + 1, c->d_counts + C_HOOK_NSEL, sizeof(int), cudaMemcpyDeviceToHost, s));
                CUDA_TRY(cudaStreamSynchronize(s));
                h_vox[2 * sg] = at; at += h_vox[2 * sg + 1];
                c->launches += c->vg.last_launches;
            }
            h_vox[2 * S] = at;
        }
    } else {
        std::memset(h_vox, 0, (size_t)(2 * S + 2) * sizeof(int));
    }
    const int n_vox = h_vox[2 * S];
    // ---- guards (:655-656); the pairs that run get the single-pair call's block partition ----
    std::vector<IcpPairDesc> pd; std::vector<int> slot_of;       // slot_of[q] = the wave's pair j
    int blocks_total = 0, tgt_total = 0;
    for (int j = 0; j < W; ++j) {
        liorf_icp_result* o = out[j];
        std::memset(o, 0, sizeof(*o));
        for (int i = 0; i < 4; ++i) o->transform[5 * i] = 1.f;
        const int so = h_vox[4 * j], sn = h_vox[4 * j + 1], to = h_vox[4 * j + 2], tn = h_vox[4 * j + 3];
        o->n_source = sn; o->n_target = tn;
        if (sn < 300 || tn < 1000) continue;
        IcpPairDesc d;
        d.src_off = so; d.n_src = sn; d.tgt_off = to; d.n_tgt = tn; d.tgt_first = tgt_total; d.part_off = blocks_total; d.pad = 0;
        d.blocks = (sn + ICP_BLOCK - 1) / ICP_BLOCK; if (d.blocks > 4 * c->num_sms) d.blocks = 4 * c->num_sms;
        blocks_total += d.blocks; tgt_total += tn;
        pd.push_back(d); slot_of.push_back(j);
    }
    const int R = (int)pd.size();
    if (R == 0) return LIORF_OK;
    // ---- per-pair target grids in one pass ----
    const GridDims g = c->icp_grid.dims;                           // the single-pair call's torus (icp_batch.cuh: why not smaller)
    const int NC = grid_cells(g);
    IcpPairDesc* h_pd = reinterpret_cast<IcpPairDesc*>(H + o_pd);
    int2* h_act = reinterpret_cast<int2*>(H + o_act);               // [0, R) every pair (fitness), [R, 2 R) the pairs still running
    IcpState* h_st = reinterpret_cast<IcpState*>(H + o_st);
    IcpState* h_stb = reinterpret_cast<IcpState*>(H + o_stb);
    double* h_fit = reinterpret_cast<double*>(H + o_fit);
    std::memcpy(h_pd, pd.data(), (size_t)R * sizeof(IcpPairDesc));
    for (int q = 0; q < R; ++q) { h_act[q] = make_int2(q, pd[q].part_off); h_act[R + q] = h_act[q]; h_st[q] = icp_initial_state(max_iters); }
    if ((rc = B.pd.reserve(R)) || (rc = B.act.reserve((size_t)2 * R)) || (rc = B.st.reserve(R)) || (rc = B.fit.reserve((size_t)2 * R)) ||
        (rc = B.partial.reserve((size_t)blocks_total * ICP_NSUM)) || (rc = reserve_zeroed(B.counters, R, s)) || (rc = reserve_zeroed(B.counts, (size_t)R * NC, s)) ||
        (rc = B.cell_start.reserve((size_t)R * NC + 1)) || (rc = B.sorted.reserve(tgt_total)) || (rc = B.src_cur.reserve(n_vox))) return rc;
    const int gtiles = (int)(((size_t)R * NC + GSCAN_TILE - 1) / GSCAN_TILE);
    if ((rc = reserve_zeroed(B.grid_scan.status, gtiles, s))) return rc;
    CUDA_TRY(cudaMemcpyAsync(B.pd.p, h_pd, (size_t)R * sizeof(IcpPairDesc), cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(B.act.p, h_act, (size_t)2 * R * sizeof(int2), cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(B.st.p, h_st, (size_t)R * sizeof(IcpState), cudaMemcpyHostToDevice, s));
    k_icpb_grid_count<<<(tgt_total + 255) / 256, 256, 0, s>>>(B.vox.p, B.pd.p, R, tgt_total, g, B.counts.p);
    k_grid_scan<<<gtiles, GSCAN_BLOCK, 0, s>>>(B.counts.p, B.cell_start.p, R * NC, B.grid_scan.ticket, B.grid_scan.status.p, B.grid_scan.err_flag);
    k_icpb_grid_scatter<<<(tgt_total + 255) / 256, 256, 0, s>>>(B.vox.p, B.pd.p, R, tgt_total, g, B.counts.p, B.cell_start.p, B.sorted.p);
    CUDA_TRY(cudaMemcpyAsync(B.src_cur.p, B.vox.p, (size_t)n_vox * sizeof(float4), cudaMemcpyDeviceToDevice, s));
    c->launches += 3;
    // ---- the ICP loops: one launch per iteration over every pair still running, read back once per chunk ----
    const int r_max = (int)std::ceil(max_corr_dist) + 1;
    const float max_d2 = max_corr_dist * max_corr_dist;
    int n_act = R, act_blocks = blocks_total, enq = 0;
    while (n_act > 0 && enq < max_iters) {
        const int todo = std::min(ICP_CHUNK, max_iters - enq);
        for (int k = 0; k < todo; ++k)
            k_icpb_iteration<<<act_blocks, ICP_BLOCK, 0, s>>>(B.pd.p, B.act.p + R, n_act, B.src_cur.p, B.st.p, B.cell_start.p, B.sorted.p, g, r_max, max_d2,
                                                              B.partial.p, B.counters.p);
        CUDA_TRY(cudaGetLastError());
        enq += todo; c->launches += todo;
        CUDA_TRY(cudaMemcpyAsync(h_stb, B.st.p, (size_t)R * sizeof(IcpState), cudaMemcpyDeviceToHost, s));
        CUDA_TRY(cudaStreamSynchronize(s));                                    // one per chunk
        n_act = 0; act_blocks = 0;
        for (int q = 0; q < R; ++q)
            if (!h_stb[q].done) { h_act[R + n_act++] = make_int2(q, act_blocks); act_blocks += pd[q].blocks; }
        if (n_act > 0 && enq < max_iters) CUDA_TRY(cudaMemcpyAsync(B.act.p + R, h_act + R, (size_t)n_act * sizeof(int2), cudaMemcpyHostToDevice, s));
    }
    // ---- getFitnessScore of every pair that ran ----
    k_icpb_fitness<<<blocks_total, ICP_BLOCK, 0, s>>>(B.pd.p, B.act.p, R, B.vox.p, B.st.p, B.cell_start.p, B.sorted.p, g, 64, B.partial.p, B.counters.p, B.fit.p);
    CUDA_TRY(cudaGetLastError());
    ++c->launches;
    CUDA_TRY(cudaMemcpyAsync(h_fit, B.fit.p, (size_t)2 * R * sizeof(double), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));                                        // the fitness sums
    for (int q = 0; q < R; ++q) icp_fill_result(h_stb[q], h_fit + 2 * q, out[slot_of[q]]);
    return LIORF_OK;
}

int liorf_loop_closure_icp_batch(liorf_ctx* c, const int* loop_key_cur, const int* loop_key_pre, const int* loop_index, int n_pairs, int history_search_num,
                                 float icp_leaf, float max_corr_dist, int max_iters, liorf_icp_result* out) {
    LIORF_NVTX;
    if (!c || n_pairs < 0 || (n_pairs > 0 && (!loop_key_cur || !loop_key_pre || !loop_index || !out))) return LIORF_ERR_ARG;
    if (history_search_num < 0 || max_iters < 1 || !(icp_leaf > 0.f) || !(max_corr_dist > 0.f)) return LIORF_ERR_ARG;
    const int n_kf = (int)c->kfs.size();
    std::vector<IcpbPair> P(n_pairs);
    for (int p = 0; p < n_pairs; ++p) {
        const int cur = loop_key_cur[p], pre = loop_key_pre[p], li = loop_index[p];
        if (cur < 0 || cur >= n_kf || pre < 0 || pre >= n_kf || li < -1 || li >= n_kf) return LIORF_ERR_ARG;
        IcpbPair& q = P[p]; q.cur = cur; q.pre = pre; q.li = li; q.raw_src = 0; q.raw_tgt = 0;
        icp_select(c, cur, 0, li, nullptr, q.raw_src);
        icp_select(c, pre, history_search_num, li, nullptr, q.raw_tgt);
        if (q.raw_src > 0x7fffffffLL || q.raw_tgt > 0x7fffffffLL || q.raw_src + q.raw_tgt > 0x7fffffffLL) return LIORF_ERR_ARG;     // as the single-pair call
    }
    if (n_pairs == 0) return LIORF_OK;
    CUDA_TRY(cudaSetDevice(c->P.device));
    int rc;
    if ((rc = join_map(c))) return rc;
    // waves: consecutive pairs while their work buffers fit the budget (a pair larger than the budget runs alone)
    std::vector<std::pair<int, int>> waves;
    {
        const int cap = c->icpb.max_pairs > 0 ? std::min(c->icpb.max_pairs, ICPB_MAX_PAIRS) : ICPB_MAX_PAIRS;
        int b = 0; size_t bytes = 0; long long pts = 0;
        for (int p = 0; p < n_pairs; ++p) {
            const long long pp = P[p].raw_src + P[p].raw_tgt;
            const size_t pb = (size_t)pp * ICPB_BYTES_PER_POINT + ICPB_GRID_BYTES;
            if (p > b && (p - b >= cap || bytes + pb > ICPB_WAVE_BYTES || pts + pp > 0x7fffffffLL)) { waves.push_back({b, p}); b = p; bytes = 0; pts = 0; }
            bytes += pb; pts += pp;
        }
        waves.push_back({b, n_pairs});
    }
    std::vector<liorf_icp_result> res(n_pairs);
    std::vector<liorf_icp_result*> res_ptr(n_pairs);
    for (int p = 0; p < n_pairs; ++p) res_ptr[p] = &res[p];
    for (size_t w = 0; w < waves.size(); ++w) {
        const int b = waves[w].first, e = waves[w].second;
        int split = 0;
        if ((rc = icpb_wave(c, P.data() + b, e - b, res_ptr.data() + b, history_search_num, icp_leaf, max_corr_dist, max_iters, &split))) return rc;
        if (split) {                                   // the wave's voxel keys need more than 32 bits: run it as two
            const int m = b + (e - b) / 2;
            waves.insert(waves.begin() + w + 1, {{b, m}, {m, e}});
        }
    }
    if ((rc = check_err(c))) return rc;
    std::memcpy(out, res.data(), (size_t)n_pairs * sizeof(liorf_icp_result));
    return LIORF_OK;
}
/* tests: at most max_pairs pairs per wave (0 = the memory-bounded default) */
int liorf_debug_icp_batch_wave(liorf_ctx* c, int max_pairs) {
    if (!c || max_pairs < 0) return LIORF_ERR_ARG;
    c->icpb.max_pairs = max_pairs;
    return LIORF_OK;
}


// ------------------------------------------------------------------------------------------------ global map (§8f-4)
// publishGlobalMap (:453-502): key poses within search_radius of the newest, thinned to pose_density voxels, nearest-1 id
// recovery, distance gate, then the selected keyframe clouds transformed by their own poses, concatenated and VoxelGrid(leaf).
// search_radius <= 0 selects EVERY keyframe (saveMapService, :379-432; leaf <= 0 there means "no down-sampling").
int liorf_build_global_map(liorf_ctx* c, float search_radius, float pose_density, float leaf, liorf_point* out, int capacity, int* n_out) {
    LIORF_NVTX;
    if (!c || !n_out || capacity < 0 || (capacity > 0 && !out)) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    *n_out = 0;
    if (c->kfs.empty()) return LIORF_OK;
    int rc;
    if ((rc = join_map(c))) return rc;
    std::vector<int> ids;
    if (search_radius > 0.f) {
        if (!(pose_density > 0.f)) return LIORF_ERR_ARG;
        std::vector<liorf_host::KeyPose> kp(c->kfs.size());
        for (size_t i = 0; i < kp.size(); ++i) { const Keyframe& k = c->kfs[i]; kp[i] = liorf_host::KeyPose{k.pose[0], k.pose[1], k.pose[2], k.pose[3], k.pose[4], k.pose[5], k.time}; }
        ids = liorf_host::extract_nearby(kp, 0.0, search_radius, pose_density, false);
    } else { ids.resize(c->kfs.size()); for (size_t i = 0; i < ids.size(); ++i) ids[i] = (int)i; }
    std::vector<KfSel> sel; long long total = 0;
    for (int id : ids) {
        const Keyframe& k = c->kfs[id];
        KfSel s; s.src_off = (int)k.off; s.count = k.count; s.dst_off = (int)total; s.pad = 0;
        host_get_transformation(k.pose[3], k.pose[4], k.pose[5], k.pose[0], k.pose[1], k.pose[2], s.t);
        total += k.count; sel.push_back(s);
    }
    if (total == 0) return LIORF_OK;
    if (total > 0x7fffffffLL) return LIORF_ERR_ARG;
    const int tot = (int)total, ns = (int)sel.size();
    if ((rc = c->icp_sel.reserve(ns)) || (rc = c->icp_raw.reserve(tot)) || (rc = c->icp_tgt.reserve(tot))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->icp_sel.p, sel.data(), (size_t)ns * sizeof(KfSel), cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    k_transform_concat<<<(tot + 255) / 256, 256, 0, c->stream>>>(c->kf_points.p, c->icp_sel.p, ns, tot, c->icp_raw.p);
    const float4* result = c->icp_raw.p; int n = tot;
    if (leaf > 0.f) {
        if ((rc = voxel_grid_device(c->icp_raw.p, Count::of_host(tot), leaf, c->icp_tgt.p, c->d_counts + C_HOOK_NSEL, nullptr, nullptr, c->vg, c->stream))) return rc;
        CUDA_TRY(cudaMemcpyAsync(c->h_mail.p + 900, c->d_counts + C_HOOK_NSEL, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        CUDA_TRY(cudaStreamSynchronize(c->stream));
        n = c->h_mail.p[900]; result = c->icp_tgt.p;
    }
    c->launches += 10;
    *n_out = n;
    if (out && n > 0) {
        if (n > capacity) return LIORF_ERR_ARG;                      // *n_out tells the caller how much room is needed
        CUDA_TRY(cudaMemcpyAsync(out, result, (size_t)n * sizeof(float4), cudaMemcpyDeviceToHost, c->stream));
    }
    return check_err(c);
}

// cloudHandler + downsampleCurrentScan of a FUTURE frame into the alternate front set, on stream_pre.
static int front_prefetch(liorf_ctx* c, const liorf_frame_in* nx) {
    if (!nx || nx->n < 0) return LIORF_ERR_ARG;
    c->pre_valid = false;
    front_swap(c);                                   // the enqueue helpers below work on "the current set" and "the context's stream"
    { int rcs = need_stream_pre(c); if (rcs) return rcs; }
    std::swap(c->stream, c->stream_pre);            // until the swap back below, c->stream is the look-ahead stream
    int rc = LIORF_OK;
    // the set being overwritten was last read by work enqueued on the main stream before this frame began (keyframe copy, ScanContext)
    if (c->frame_start_recorded && cudaStreamWaitEvent(c->stream, c->ev_frame_start, 0) != cudaSuccess) rc = LIORF_ERR_CUDA;
    if (!rc) {
        if (nx->pts_on_device) rc = liorf_project_point_cloud_dev(c, nx->pts, nx->n, nx->time_scan_cur, nx->imu_time, nx->imu_rot_x, nx->imu_rot_y, nx->imu_rot_z,
                                                                  nx->imu_pointer_cur, nx->deskew_enabled);
        else rc = liorf_project_point_cloud(c, (const liorf_point_xyzirt*)nx->pts, nx->n, nx->time_scan_cur, nx->imu_time, nx->imu_rot_x, nx->imu_rot_y,
                                            nx->imu_rot_z, nx->imu_pointer_cur, nx->deskew_enabled, nullptr, nullptr, nullptr);
    }
    if (!rc) rc = downsample_async(c, nullptr, c->num_sms - c->s2m_grid >= 4 ? c->num_sms - c->s2m_grid : 0);      // beside the solver: its spare SMs
    if (!rc && cudaEventRecord(c->ev_pre_done, c->stream) != cudaSuccess) rc = LIORF_ERR_CUDA;
    std::swap(c->stream, c->stream_pre);
    front_swap(c);
    if (rc) return rc;
    c->pre_valid = true; c->pre_index = nx->frame_index; c->pre_n = nx->n; c->pre_pts = nx->pts;
    return LIORF_OK;
}

int liorf_cloud_handler_async(liorf_ctx* c, const liorf_frame_in* frame) {
    LIORF_NVTX;
    if (!c || !frame) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    CUDA_TRY(cudaEventRecord(c->ev_frame_start, c->stream)); c->frame_start_recorded = true;
    return front_prefetch(c, frame);
}

int liorf_process_frame(liorf_ctx* c, const liorf_frame_in* in, liorf_frame_out* out) {
    LIORF_NVTX;
    if (!c || !in || !out || in->n < 0) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    int rc;
    std::memset(out, 0, sizeof(*out)); out->keyframe_id = -1; out->loop_id = -1;
    using clk = std::chrono::steady_clock;
    auto T0 = clk::now();
    auto stamp = [&](int k, cudaStream_t st) { if (c->host_timing) { if (!c->tl_ev[k]) (void)event_create(c->tl_ev[k], cudaEventDefault); cudaEventRecord(c->tl_ev[k], st); } };
    stamp(0, c->stream);
    auto lap = [&](int k) { if (c->host_timing) { auto t = clk::now(); c->host_us[k] += std::chrono::duration<double, std::micro>(t - T0).count(); T0 = t; } };
    // everything the earlier frames left on the main stream precedes this point: the front set they lived in may be refilled after it
    CUDA_TRY(cudaEventRecord(c->ev_frame_start, c->stream)); c->frame_start_recorded = true;
    // cloudHandler: projectPointCloud (the deskewed cloud stays on the device) — already done on stream_pre when this frame was
    // announced as the previous call's `next` (or through liorf_cloud_handler_async)
    const bool prefetched = c->pre_valid && c->pre_index == in->frame_index && c->pre_n == in->n && c->pre_pts == in->pts;
    c->pre_valid = false;
    if (prefetched) {
        front_swap(c);
        CUDA_TRY(cudaStreamWaitEvent(c->stream, c->ev_pre_done, 0));
    } else {
        if (in->pts_on_device) rc = liorf_project_point_cloud_dev(c, in->pts, in->n, in->time_scan_cur, in->imu_time, in->imu_rot_x, in->imu_rot_y, in->imu_rot_z,
                                                                  in->imu_pointer_cur, in->deskew_enabled);
        else rc = liorf_project_point_cloud(c, (const liorf_point_xyzirt*)in->pts, in->n, in->time_scan_cur, in->imu_time, in->imu_rot_x, in->imu_rot_y, in->imu_rot_z,
                                            in->imu_pointer_cur, in->deskew_enabled, nullptr, nullptr, nullptr);
        if (rc) return rc;
    }
    stamp(1, c->stream);
    lap(0);
    // laserCloudInfoHandler: extractSurroundingKeyFrames, downsampleCurrentScan, scan2MapOptimization.  The local-map chain is the
    // longer of the two independent preparations, so it is enqueued first (on its own stream); the downsample follows on the
    // main stream while it runs.
    if (!c->kfs.empty()) {
        std::vector<liorf_host::KeyPose> kp(c->kfs.size());
        for (size_t i = 0; i < kp.size(); ++i) { const Keyframe& k = c->kfs[i]; kp[i] = liorf_host::KeyPose{k.pose[0], k.pose[1], k.pose[2], k.pose[3], k.pose[4], k.pose[5], k.time}; }
        std::vector<int> sel = liorf_host::extract_nearby(kp, in->time_scan_cur, c->P.surroundingKeyframeSearchRadius, in->surrounding_keyframe_density);
        if ((rc = liorf_extract_surrounding_keyframes(c, sel.data(), (int)sel.size(), nullptr))) return rc;
    }
    stamp(2, c->stream_map ? c->stream_map : c->stream);
    lap(1);
    if (!prefetched && (rc = liorf_downsample_current_scan(c, nullptr, nullptr, nullptr))) return rc;
    stamp(3, c->stream);
    lap(2);
    if ((rc = join_map(c))) return rc;
    stamp(4, c->stream);
    float guess[6];
    if (in->use_cloud_info) {                                                    // updateInitialGuess (:899-958) from the previous pose
        std::memcpy(guess, c->tf_mapped, sizeof(guess));
        liorf_host_update_initial_guess(&c->guess_state, c->kfs.empty() ? 1 : 0, &in->cloud_info, in->use_imu_heading_initialization, in->imu_type, guess);
    } else std::memcpy(guess, in->initial_guess, sizeof(guess));
    if ((rc = launch_s2m(c, in->max_iters > 0 ? in->max_iters : 30, 0, true, guess))) return rc;
    stamp(5, c->stream);
    // the NEXT frame's cloudHandler + downsample go to stream_pre now, behind this frame's critical chain in host order, and run
    // on the device while the solver iterates (the reference runs imageProjection and mapOptimization as two concurrent nodes)
    if (in->next && (rc = front_prefetch(c, (const liorf_frame_in*)in->next))) return rc;
    lap(3);
    if ((rc = get_pose_mail(c, out->pose, &out->iters, &out->converged, &out->degenerate, &out->ran))) return rc;   // the frame's single round trip
    lap(4);
    if (c->host_timing) for (int k = 1; k <= 5; ++k) { float ms = 0; if (c->tl_ev[k] && cudaEventElapsedTime(&ms, c->tl_ev[0], c->tl_ev[k]) == cudaSuccess) c->tl_ms[k] += ms; }
    out->n_kept = c->h_n_scan; out->n_ds = c->h_n_ds; out->m_ds = c->h_m_ds;
    if (out->ran) {                                                              // transformUpdate (:1323-1353) only after a solve (:1317)
        if (in->use_cloud_info) liorf_host::transform_update(out->pose, in->cloud_info.imuAvailable != 0, in->imu_type, in->cloud_info.imuRollInit,
                                                             in->cloud_info.imuPitchInit, in->imu_rpy_weight, in->rotation_tollerance, in->z_tollerance);
        else liorf_host::transform_update_clamp(out->pose, in->rotation_tollerance, in->z_tollerance);
    }
    std::memcpy(c->tf_mapped, out->pose, sizeof(c->tf_mapped));
    // saveKeyFramesAndFactor (the parts on the path): saveFrame gate, keyframe cloud, ScanContext descriptor
    auto T1 = clk::now();
    auto sub = [&](int k) { if (c->host_timing) { auto t = clk::now(); c->host_us[k] += std::chrono::duration<double, std::micro>(t - T1).count(); T1 = t; } };
    if (liorf_save_frame(c, out->pose, in->adding_dist_threshold, in->adding_angle_threshold) == 1) {
        int id = liorf_add_keyframe(c, out->pose, in->time_scan_cur);
        if (id < 0) return id;
        out->is_keyframe = 1; out->keyframe_id = id;
        sub(6);
        // A new keyframe changes the NEXT frame's local map.  With look-ahead its timestamp is known, so extractSurroundingKeyFrames
        // for that frame is launched right here (stream_map, behind the keyframe copy only) instead of after the host has returned,
        // built the next call and come back; the next call's identical request then finds the map resident.
        if (in->next) {
            const liorf_frame_in* nx = (const liorf_frame_in*)in->next;
            std::vector<liorf_host::KeyPose> kp(c->kfs.size());
            for (size_t i = 0; i < kp.size(); ++i) { const Keyframe& k = c->kfs[i]; kp[i] = liorf_host::KeyPose{k.pose[0], k.pose[1], k.pose[2], k.pose[3], k.pose[4], k.pose[5], k.time}; }
            std::vector<int> sel = liorf_host::extract_nearby(kp, nx->time_scan_cur, c->P.surroundingKeyframeSearchRadius, nx->surrounding_keyframe_density);
            sub(7);
            if ((rc = liorf_extract_surrounding_keyframes(c, sel.data(), (int)sel.size(), nullptr))) return rc;
            sub(8);
        }
        if ((rc = liorf_sc_make_and_save(c, nullptr, 0))) return rc;
        sub(9);
    }
    if (in->loop_every > 0 && in->frame_index % in->loop_every == in->loop_every - 1) {
        out->loop_checked = 1;
        if ((rc = liorf_sc_detect_loop_closure_id(c, &out->loop_id, &out->loop_yaw, nullptr, nullptr))) return rc;
        sub(10);
    }
    lap(5); ++c->host_frames;
    return LIORF_OK;
}

// Pre-sizes every work buffer so that no call allocates afterwards (allocation = cudaMalloc/cudaFree = device sync).
int liorf_reserve(liorf_ctx* c, int n_scan_max, int m_raw_max, int n_keyframe_points_max, int sc_entries_max) {
    LIORF_NVTX;
    if (!c || n_scan_max < 0 || m_raw_max < 0) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    if (c->stream_pre) CUDA_TRY(cudaStreamSynchronize(c->stream_pre)); c->pre_valid = false;
    int rc;
    const size_t n = (size_t)(n_scan_max > 0 ? n_scan_max : 1), m = (size_t)(m_raw_max > 0 ? m_raw_max : 1), big = n > m ? n : m;
    for (int set = 0; set < 2; ++set) {                           // both front sets (see liorf_ctx::FrontSet)
        rc = 0;
        if ((rc = c->scan.reserve(n)) || (rc = c->scan_ds.reserve(n)) || (rc = c->dk.raw.reserve(n)) || (rc = c->dk.kept.reserve(n)) ||
            (rc = c->vg.keys.reserve(big)) || (rc = c->vg.seg_start.reserve(big + 1)) || (rc = c->vg.partial.reserve((size_t)kNumSMs * 6)) ||
            (rc = c->vg.sort.keys_alt.reserve(big)) || (rc = c->vg.sort.vals_a.reserve(big)) || (rc = c->vg.sort.vals_b.reserve(big)) ||
            (rc = c->vg.sort.hist.reserve(4 * RADIX)) ||
            (rc = reserve_zeroed(c->vg.sort.status, ((big + SORT_TILE - 1) / SORT_TILE) * RADIX, c->stream)) ||
            (rc = reserve_zeroed(c->vg.scan.status, (big + SCAN_TILE - 1) / SCAN_TILE, c->stream)) ||
            (rc = reserve_zeroed(c->dk.scan.status, (n + SCAN_TILE - 1) / SCAN_TILE, c->stream))) { /* fall through to the swap back */ }
        front_swap(c);
        if (rc && set == 0) { front_swap(c); return rc; }
        if (rc) return rc;
    }
    if ((rc = c->membership.reserve(big)) || (rc = c->out_keys.reserve(big)) ||
        (rc = c->map_raw.reserve(m)) || (rc = c->map_ds.reserve(m)) || (rc = c->grid.sorted.reserve(m)) ||
        (rc = c->qcache.reserve(n)) || (rc = c->cand.reserve((size_t)n * S2M_GROW)) || (rc = c->d_sel.reserve(4096)) ||
        (rc = c->vg_map.keys.reserve(m)) || (rc = c->vg_map.seg_start.reserve(m + 1)) || (rc = c->vg_map.partial.reserve((size_t)kNumSMs * 6)) ||
        (rc = c->vg_map.sort.keys_alt.reserve(m)) || (rc = c->vg_map.sort.vals_a.reserve(m)) || (rc = c->vg_map.sort.vals_b.reserve(m)) ||
        (rc = c->vg_map.sort.hist.reserve(4 * RADIX)) ||
        (rc = reserve_zeroed(c->vg_map.sort.status, ((m + SORT_TILE - 1) / SORT_TILE) * RADIX, c->stream)) ||
        (rc = reserve_zeroed(c->vg_map.scan.status, (m + SCAN_TILE - 1) / SCAN_TILE, c->stream))) return rc;
    if (n_keyframe_points_max > 0 && (rc = c->kf_points.reserve((size_t)n_keyframe_points_max, c->stream, true))) return rc;
    if (sc_entries_max > 0 && (rc = sc_reserve(c, sc_entries_max))) return rc;
    if ((rc = c->h_sel.reserve((size_t)2 * 4096))) return rc;
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return LIORF_OK;
}

// ---- benchmark / introspection helpers ----
int liorf_enable_timing(liorf_ctx* c, int on) {
    LIORF_NVTX;
    if (!c) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    CUDA_TRY(cudaStreamSynchronize(c->stream)); prof_flush(c);
    c->prof.enabled = on != 0; c->prof.mask = 0xffu;
    for (int i = 0; i < SEC_COUNT; ++i) { c->prof.ms[i] = 0; c->prof.calls[i] = 0; }
    return LIORF_OK;
}
/* like liorf_enable_timing(ctx, 1) but only the sections whose bit is set in `mask` record events (two cudaEventRecord calls per
 * section and frame are host time on the frame's critical path: the headline window times the dominant kernel only) */
int liorf_enable_timing_mask(liorf_ctx* c, unsigned mask) {
    LIORF_NVTX;
    int rc = liorf_enable_timing(c, mask != 0);
    if (!rc) c->prof.mask = mask & 0xffu;
    return rc;
}
int liorf_get_timing(liorf_ctx* c, double ms[8], long long calls[8]) {
    LIORF_NVTX;
    if (!c || !ms || !calls) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    CUDA_TRY(cudaStreamSynchronize(c->stream)); prof_flush(c);
    for (int i = 0; i < SEC_COUNT; ++i) { ms[i] = c->prof.ms[i]; calls[i] = c->prof.calls[i]; }
    return LIORF_OK;
}
long long liorf_get_launch_count(liorf_ctx* c) { return c ? c->launches : -1; }
// debug: phase clocks of the persistent solver (CTA 0): out[iter*8 + {0 start,1 loop done,2 block reduced,3 grid synced,4 summed,5 solved}]
/* tests: 1 = the solver never reuses its per-query candidate lists / plane fits (reference-style full search every iteration) */
int liorf_debug_s2m_disable_cache(liorf_ctx* c, int on) {
    LIORF_NVTX;
    if (!c) return LIORF_ERR_ARG;
    c->s2m_no_cache = on != 0;
    return LIORF_OK;
}
/* tests: 1 = the solver keeps its per-query state (cache header, candidate list) in global memory even when the scan fits one round
 * of the grid (the layout multi-round solves use); 0 = automatic (shared memory whenever one round covers the scan) */
int liorf_debug_s2m_global_state(liorf_ctx* c, int on) {
    LIORF_NVTX;
    if (!c) return LIORF_ERR_ARG;
    c->s2m_global_state = on != 0;
    return LIORF_OK;
}
/* tests: the solver runs on `ctas` CTAs (ctas - 1 workers and the reducer) in every launch, per-function calls and liorf_process_frame
 * alike, so that each layout of k_scan2map_persistent can be reached on any scan size; 0 = the defaults.  The cooperative launch needs
 * every CTA resident at once, one per SM: 2 <= ctas <= num_sms.  The front end's share of the SMs in liorf_process_frame does not change. */
int liorf_debug_s2m_grid(liorf_ctx* c, int ctas) {
    LIORF_NVTX;
    if (!c || (ctas != 0 && (ctas < 2 || ctas > c->num_sms))) return LIORF_ERR_ARG;
    c->s2m_ctas = ctas;
    return LIORF_OK;
}
/* debug: %globaltimer stamps of the last solve, out[iter * 160 + k]: k < workers = that worker's arrival, 156 = reducer sums
 * ready, 157 = reducer published, 158 = worker 0 saw the flag (ns) */
int liorf_debug_s2m_arrivals(liorf_ctx* c, int enable, unsigned long long* out /* 64*160 or null */) {
    LIORF_NVTX;
    if (!c) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    const size_t bytes = (size_t)S2M_MAX_ITERS * S2M_GT_STRIDE * sizeof(unsigned long long);
    if (enable && !c->d_dbg_gt) { CUDA_TRY(dev_alloc(c->d_dbg_gt, (size_t)S2M_MAX_ITERS * S2M_GT_STRIDE)); CUDA_TRY(cudaMemset(c->d_dbg_gt, 0, bytes)); }
    if (out && c->d_dbg_gt) CUDA_TRY(cudaMemcpy(out, c->d_dbg_gt, bytes, cudaMemcpyDeviceToHost));
    if (!enable) c->d_dbg_gt.reset();
    return LIORF_OK;
}
int liorf_debug_s2m_clocks(liorf_ctx* c, int enable, long long* out /*64*8 or null*/) {
    LIORF_NVTX;
    if (!c) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    if (enable && !c->d_dbg) { CUDA_TRY(dev_alloc(c->d_dbg, S2M_MAX_ITERS * 8)); CUDA_TRY(cudaMemset(c->d_dbg, 0, S2M_MAX_ITERS * 8 * sizeof(long long))); }
    if (out && c->d_dbg) CUDA_TRY(cudaMemcpy(out, c->d_dbg, S2M_MAX_ITERS * 8 * sizeof(long long), cudaMemcpyDeviceToHost));
    if (!enable) c->d_dbg.reset();
    return LIORF_OK;
}
int liorf_get_last_counts(liorf_ctx* c, int* n_scan, int* n_ds, int* m_ds, int* iters) {
    LIORF_NVTX;
    if (!c) return LIORF_ERR_ARG;
    if (n_scan) *n_scan = c->rep_counts[0]; if (n_ds) *n_ds = c->rep_counts[1]; if (m_ds) *m_ds = c->rep_counts[2];
    if (iters) *iters = c->h_mail.p[1024 + 448];       // S2MTrace.iters as of the last liorf_get_pose
    return LIORF_OK;
}
int liorf_get_keyframe(liorf_ctx* c, int id, liorf_point* out, int capacity, int* n, float pose6[6], double* time) {
    LIORF_NVTX;
    if (!c || id < 0 || id >= (int)c->kfs.size()) return LIORF_ERR_ARG;
    CUDA_TRY(cudaSetDevice(c->P.device));
    const Keyframe& k = c->kfs[id];
    if (n) *n = k.count;
    if (pose6) std::memcpy(pose6, k.pose, 6 * sizeof(float));
    if (time) *time = k.time;
    if (out) {
        if (capacity < k.count) return LIORF_ERR_ARG;
        CUDA_TRY(cudaStreamSynchronize(c->stream));
        if (k.count > 0) CUDA_TRY(cudaMemcpy(out, c->kf_points.p + k.off, (size_t)k.count * sizeof(float4), cudaMemcpyDeviceToHost));
    }
    return LIORF_OK;
}

}  // extern "C"
