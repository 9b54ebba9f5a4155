// common.cuh — shared types and helpers of the B200 (sm_100a) scan-to-map library.
// The whole library is compiled with -fmad=false: parity-critical fp32 expressions keep the
// reference's operation order (x86-64 baseline build, no FMA: CMakeLists.txt:7).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cmath>
#include <memory>
#include <utility>

#define LIORF_OK 0
#define LIORF_ERR_CUDA -1
#define LIORF_ERR_ARG -2
#define LIORF_ERR_STATE -3
#define LIORF_ERR_DEVICE_FLAG -4

#define CUDA_TRY(expr)                                                                       \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            fprintf(stderr, "[liorf_b200] CUDA error %s at %s:%d: %s\n", cudaGetErrorName(_e), __FILE__, __LINE__, \
                    cudaGetErrorString(_e));                                                 \
            return LIORF_ERR_CUDA;                                                           \
        }                                                                                    \
    } while (0)

namespace liorf {

constexpr int kNumSMs = 148;          // B200: 2 dies x 74 SMs; grids are sized in multiples of this
constexpr unsigned FULL = 0xffffffffu;

// Every CUDA resource a context acquires is held by one of the owners below, which release it when they are destroyed.  They are
// move-only.  An Owned converts to its raw handle, so call sites use it like the handle; a raw copy of a handle is a view and must not
// outlive its owner.  An acquire helper replaces what the owner held only when the call returned a handle.
template <auto Release> struct Releaser { template <class H> void operator()(H h) const { Release(h); } };
template <class T, auto Release>
struct Owned : std::unique_ptr<T, Releaser<Release>> {
    using std::unique_ptr<T, Releaser<Release>>::unique_ptr;
    operator T*() const { return this->get(); }
};
template <class T> using DevMem = Owned<T, cudaFree>;                    // fixed-size device allocation
template <class T> using IpcMapping = Owned<T, cudaIpcCloseMemHandle>;   // another process's allocation mapped into this one
using Stream = Owned<CUstream_st, cudaStreamDestroy>;
using Event = Owned<CUevent_st, cudaEventDestroy>;
using Graph = Owned<CUgraph_st, cudaGraphDestroy>;
using GraphExec = Owned<CUgraphExec_st, cudaGraphExecDestroy>;

template <class O, class F> cudaError_t acquire(O& o, F&& get) {
    typename O::pointer h = nullptr;
    const cudaError_t e = get(&h);
    if (h) o.reset(h);           // also a graph that cudaStreamEndCapture returns together with an error
    return e;
}
template <class T> cudaError_t dev_alloc(DevMem<T>& m, size_t n) { return acquire(m, [&](T** h) { return cudaMalloc(h, n * sizeof(T)); }); }
inline cudaError_t stream_create(Stream& s, int priority) {
    return acquire(s, [&](cudaStream_t* h) { return cudaStreamCreateWithPriority(h, cudaStreamNonBlocking, priority); });
}
inline cudaError_t event_create(Event& ev, unsigned flags) { return acquire(ev, [&](cudaEvent_t* h) { return cudaEventCreateWithFlags(h, flags); }); }
inline cudaError_t end_capture(Graph& g, cudaStream_t s) { return acquire(g, [&](cudaGraph_t* h) { return cudaStreamEndCapture(s, h); }); }
inline cudaError_t graph_instantiate(GraphExec& x, cudaGraph_t g) { return acquire(x, [&](cudaGraphExec_t* h) { return cudaGraphInstantiate(h, g, 0); }); }
template <class T> cudaError_t ipc_open(IpcMapping<T>& m, cudaIpcMemHandle_t handle) {
    return acquire(m, [&](T** h) { return cudaIpcOpenMemHandle(reinterpret_cast<void**>(h), handle, cudaIpcMemLazyEnablePeerAccess); });
}

// growable device buffer (capacity only grows; contents are NOT preserved across growth unless asked)
template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, 0)) {}
    DevBuf& operator=(DevBuf&& o) noexcept { if (this != &o) { release(); p = std::exchange(o.p, nullptr); cap = std::exchange(o.cap, 0); } return *this; }
    ~DevBuf() { release(); }
    int reserve(size_t n, cudaStream_t s = nullptr, bool keep = false) {
        if (n <= cap) return LIORF_OK;
        size_t ncap = cap ? cap : 1024;
        while (ncap < n) ncap = 2 * ncap + 1024;          // doubling: growth (a cudaMalloc + cudaFree sync) must stay rare
        DevMem<T> np_;
        CUDA_TRY(dev_alloc(np_, ncap));
        if (keep && p && cap) CUDA_TRY(cudaMemcpyAsync(np_, p, cap * sizeof(T), cudaMemcpyDeviceToDevice, s));
        if (p) { if (keep) CUDA_TRY(cudaStreamSynchronize(s)); CUDA_TRY(cudaFree(p)); }
        p = np_.release(); cap = ncap;
        return LIORF_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// growable pinned host buffer: grows to exactly the size asked for and keeps no contents.  The caller synchronises whatever stream may
// still copy from or to the old block before it grows.
template <class T>
struct HostBuf {
    Owned<T, cudaFreeHost> p;
    size_t cap = 0;
    HostBuf() = default;
    HostBuf(HostBuf&& o) noexcept : p(std::move(o.p)), cap(std::exchange(o.cap, 0)) {}
    HostBuf& operator=(HostBuf&& o) noexcept { p = std::move(o.p); cap = std::exchange(o.cap, 0); return *this; }
    int reserve(size_t n) {
        if (n <= cap) return LIORF_OK;
        p.reset(); cap = 0;
        T* np_ = nullptr;
        CUDA_TRY(cudaHostAlloc(&np_, n * sizeof(T), cudaHostAllocDefault));
        p.reset(np_); cap = n;
        return LIORF_OK;
    }
};

// correctly-rounded-in-practice float trig: evaluate in fp64, round once (see DESIGN.md "transcendentals")
__device__ __forceinline__ float sin_f(float x) { return (float)sin((double)x); }
__device__ __forceinline__ float cos_f(float x) { return (float)cos((double)x); }

// pcl::getTransformation (float), row-major 3x4 — mirrors oracle get_transformation
__device__ __forceinline__ void get_transformation_dev(float x, float y, float z, float roll, float pitch, float yaw, float t[12]) {
    float A = cos_f(yaw), B = sin_f(yaw), C = cos_f(pitch), D = sin_f(pitch);
    float E = cos_f(roll), F = sin_f(roll), DE = D * E, DF = D * F;
    t[0] = A * C;  t[1] = A * DF - B * E;  t[2]  = B * F + A * DE;  t[3]  = x;
    t[4] = B * C;  t[5] = A * E + B * DF;  t[6]  = B * DE - A * F;  t[7]  = y;
    t[8] = -D;     t[9] = C * F;           t[10] = C * E;           t[11] = z;
}

// pointAssociateToMap op order (src/mapOptmization.cpp:304-306)
__device__ __forceinline__ float4 apply_affine_dev(const float* __restrict__ t, float4 p) {
    float4 o;
    o.x = t[0] * p.x + t[1] * p.y + t[2]  * p.z + t[3];
    o.y = t[4] * p.x + t[5] * p.y + t[6]  * p.z + t[7];
    o.z = t[8] * p.x + t[9] * p.y + t[10] * p.z + t[11];
    o.w = p.w;
    return o;
}

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ int warp_id() { return threadIdx.x >> 5; }

}  // namespace liorf
