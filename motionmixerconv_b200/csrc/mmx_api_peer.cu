// Gradient exchange fused into the optimiser: ONE kernel per step does the all-reduce of the flat gradient bucket over
// NVLink / NVSwitch peer memory AND the Adam update (batch-sharded data parallelism, one process per GPU).
//
// The reference has no data-parallel path (single device, train_mixer_h36m.py:63,193); BASELINE.json's north star asks for
// "batch-sharded data parallelism across the 8 GPUs of one box with a bucketed gradient allreduce over NCCL/NVLink".  The
// bucket is small (K2: 120 KB, K4: 730 KB), so the exchange is latency-bound: an NCCL all-reduce launch + the Adam launch cost
// ~45 us of a 0.8 ms step and sit between two CUDA graphs.  Here every rank's gradient bucket lives in a cudaMalloc'ed,
// IPC-exported allocation that every peer maps (mmx_peer_alloc / mmx_ipc_export / mmx_ipc_open); the kernel
//   1. signals "my gradients are final" into every peer's flag block (st.release.sys through the peer mapping),
//   2. waits until every peer has signalled (ld.acquire.sys on its own flag block),
//   3. reads chunk c of EVERY rank's bucket with plain peer loads (one-shot all-reduce: W reads per element, summed in rank
//      order 0..W-1 on every rank, so all replicas compute bit-identical sums) and applies Adam to its own replica,
//   4. signals "done reading" and waits for the peers' done signals for its chunk, so the next step's memset of the bucket
//      cannot overtake a peer that is still reading it.
// CTA c only ever talks to CTA c of the peers (flag slot [phase][src rank][c]); the grid is small enough to be co-resident.
// All spins are bounded (~15 s): a rank that never arrives ends the kernel with the abort counter bumped instead of hanging.
// The kernel holds no host-visible state: the epoch lives in device memory and is advanced by the last CTA, so the whole
// training step (forward, backward, this kernel) is ONE CUDA graph.
#include "mmx_launch.cuh"

#if defined(MMX_HOST_EMU)
extern "C" int mmx_peer_alloc(long long, void**) { return fail(MMX_E_UNSUPPORTED, "mmx_peer_alloc: not in the emulator"); }
extern "C" int mmx_peer_free(void*) { return fail(MMX_E_UNSUPPORTED, "mmx_peer_free: not in the emulator"); }
extern "C" int mmx_ipc_export(void*, unsigned char*) { return fail(MMX_E_UNSUPPORTED, "mmx_ipc_export: not in the emulator"); }
extern "C" int mmx_ipc_open(const unsigned char*, void**) { return fail(MMX_E_UNSUPPORTED, "mmx_ipc_open: not in the emulator"); }
extern "C" int mmx_ipc_close(void*) { return fail(MMX_E_UNSUPPORTED, "mmx_ipc_close: not in the emulator"); }
extern "C" int mmx_peer_flag_bytes(int world) { return 2 * world * 128 * 4; }
extern "C" int mmx_adam_step_peer(float*, float*, float*, const void*, const void*, int, int, long long, const float*, unsigned int*, void*) {
    return fail(MMX_E_UNSUPPORTED, "mmx_adam_step_peer: not in the emulator");
}
#else
using namespace mmx;

namespace {

constexpr int kPeerCtas = 128;       // flag slots per rank and phase = upper bound of the grid (CTA c owns chunk c of the bucket)
constexpr int kPeerThreads = 256;
constexpr int kMaxWorld = 16;

struct PeerArgs {
    float *p, *m, *v;
    const float* const* peer_g;          // DEVICE array [world]: every rank's gradient bucket as mapped in this process
    unsigned int* const* peer_flags;     // DEVICE array [world]: every rank's flag block  [2][world][kPeerCtas]
    const float* hp;
    unsigned int* epoch;                 // DEVICE [2]: epoch of the last completed exchange, CTA completion counter
    int* abort_count;
    long long n;
    int rank, world;
    int grid;                            // CTAs of this launch (the same on every rank: a function of n only)
};

__device__ __forceinline__ void st_release_sys(unsigned int* p, unsigned int v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float4 ld_peer4(const float* p) {      // never served from a stale L1 line
    float4 v;
    asm volatile("ld.volatile.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
// spin until *flag == want; false (and *timed_out set) after ~15 s
__device__ __forceinline__ bool wait_flag(const unsigned int* flag, unsigned int want, int* timed_out) {
    const long long t0 = clock64();
    while (ld_acquire_sys(flag) != want) {
        if (clock64() - t0 > 30000000000ll) { *timed_out = 1; return false; }
        __nanosleep(32);
    }
    return true;
}

__global__ void __launch_bounds__(kPeerThreads) adam_peer_kernel(const PeerArgs a) {
    __shared__ unsigned int s_epoch;
    __shared__ int s_timeout;
    const int tid = threadIdx.x, c = blockIdx.x, W = a.world, G = kPeerCtas, NG = a.grid;
    if (tid == 0) { s_epoch = a.epoch[0] + 1u; s_timeout = 0; }
    __syncthreads();
    const unsigned int e = s_epoch;
    unsigned int* mine = a.peer_flags[a.rank];
    // ---- 1. arrive: this rank's gradients are final (they were written by earlier kernels of this stream)
    if (tid < W) st_release_sys(a.peer_flags[tid] + (0 * W + a.rank) * G + c, e);
    // ---- 2. every peer has arrived
    if (tid < W) wait_flag(mine + (0 * W + tid) * G + c, e, &s_timeout);
    __syncthreads();
    // ---- 3. one-shot all-reduce of chunk c: sums of up to kHold float4 per thread stay in registers, so that
    // ---- 4. "done reading" can be signalled BEFORE the Adam arithmetic (the peers' next memset waits on it, not on our math)
    const float lr = a.hp[0], b2 = a.hp[2], eps = a.hp[3], wd = a.hp[4];
    const float bc1 = a.hp[5], bc2s = a.hp[6], gs = a.hp[7], omb1 = a.hp[8], omb2 = a.hp[9];
    const float step = lr / bc1;
    const long long n4 = a.n >> 2, stride = (long long)NG * kPeerThreads, i0 = (long long)c * kPeerThreads + tid;
    const float* pg[kMaxWorld];
#pragma unroll
    for (int r = 0; r < kMaxWorld; ++r) pg[r] = r < W ? a.peer_g[r] : nullptr;
    auto reduce4 = [&](long long i) {
        float4 g = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
#pragma unroll
        for (int r = 0; r < kMaxWorld; ++r)
            if (r < W) {
                const float4 t = ld_peer4(pg[r] + 4 * i);
                g.x += t.x; g.y += t.y; g.z += t.z; g.w += t.w;
            }
        return g;
    };
    auto adam4 = [&](long long i, const float4 g) {
        const float4 p = *reinterpret_cast<const float4*>(a.p + 4 * i), m = *reinterpret_cast<const float4*>(a.m + 4 * i),
                     v = *reinterpret_cast<const float4*>(a.v + 4 * i);
        float pp[4] = {p.x, p.y, p.z, p.w}, gg[4] = {g.x, g.y, g.z, g.w}, mm[4] = {m.x, m.y, m.z, m.w}, vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float gr = fmaf(wd, pp[k], gs * gg[k]);
            mm[k] = mm[k] + (gr - mm[k]) * omb1;
            vv[k] = fmaf(vv[k], b2, omb2 * gr * gr);
            pp[k] -= step * (mm[k] / (sqrtf(vv[k]) / bc2s + eps));
        }
        *reinterpret_cast<float4*>(a.p + 4 * i) = make_float4(pp[0], pp[1], pp[2], pp[3]);
        *reinterpret_cast<float4*>(a.m + 4 * i) = make_float4(mm[0], mm[1], mm[2], mm[3]);
        *reinterpret_cast<float4*>(a.v + 4 * i) = make_float4(vv[0], vv[1], vv[2], vv[3]);
    };
    constexpr int kHold = 4;
    float4 held[kHold];
#pragma unroll
    for (int k = 0; k < kHold; ++k)
        if (i0 + k * stride < n4) held[k] = reduce4(i0 + k * stride);
    for (long long i = i0 + kHold * stride; i < n4; i += stride) adam4(i, reduce4(i));      // buckets above 1 M floats: the rest, fused
    __syncthreads();
    if (tid < W) st_release_sys(a.peer_flags[tid] + (1 * W + a.rank) * G + c, e);      // (the CTA's peer loads completed before the barrier)
#pragma unroll
    for (int k = 0; k < kHold; ++k)
        if (i0 + k * stride < n4) adam4(i0 + k * stride, held[k]);
    // nobody may still be reading this rank's chunk c when the kernel ends
    if (tid < W) wait_flag(mine + (1 * W + tid) * G + c, e, &s_timeout);
    __syncthreads();
    if (tid == 0) {
        if (s_timeout) atomicAdd(a.abort_count, 1);
        __threadfence();
        if (atomicAdd(a.epoch + 1, 1u) == (unsigned int)(NG - 1)) {       // the last CTA publishes the epoch for the next launch
            a.epoch[1] = 0u;
            __threadfence();
            a.epoch[0] = e;
        }
    }
}

}  // namespace

extern "C" int mmx_peer_flag_bytes(int world) { return 2 * world * kPeerCtas * 4; }

extern "C" int mmx_peer_alloc(long long bytes, void** ptr) {
    if (bytes <= 0 || !ptr) return fail(MMX_E_INVALID, "mmx_peer_alloc: bad argument");
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, (size_t)bytes);
    if (e == cudaSuccess) e = cudaMemset(p, 0, (size_t)bytes);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(MMX_E_CUDA, "mmx_peer_alloc(%lld): %s", bytes, cudaGetErrorString(e)); }
    *ptr = p;
    return MMX_OK;
}
extern "C" int mmx_peer_free(void* ptr) {
    cudaError_t e = cudaFree(ptr);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(MMX_E_CUDA, "mmx_peer_free: %s", cudaGetErrorString(e)); }
    return MMX_OK;
}
extern "C" int mmx_ipc_export(void* ptr, unsigned char* handle64) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    if (!ptr || !handle64) return fail(MMX_E_INVALID, "mmx_ipc_export: null pointer");
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, ptr);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(MMX_E_CUDA, "cudaIpcGetMemHandle: %s", cudaGetErrorString(e)); }
    memcpy(handle64, &h, 64);
    return MMX_OK;
}
extern "C" int mmx_ipc_open(const unsigned char* handle64, void** ptr) {
    if (!handle64 || !ptr) return fail(MMX_E_INVALID, "mmx_ipc_open: null pointer");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    void* p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(MMX_E_CUDA, "cudaIpcOpenMemHandle: %s", cudaGetErrorString(e)); }
    *ptr = p;
    return MMX_OK;
}
extern "C" int mmx_ipc_close(void* ptr) {
    cudaError_t e = cudaIpcCloseMemHandle(ptr);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(MMX_E_CUDA, "cudaIpcCloseMemHandle: %s", cudaGetErrorString(e)); }
    return MMX_OK;
}

extern "C" int mmx_adam_step_peer(float* p, float* m, float* v, const void* peer_g, const void* peer_flags, int rank, int world, long long n,
                                  const float* hyper, unsigned int* epoch, void* stream) {
    if (!p || !m || !v || !peer_g || !peer_flags || !hyper || !epoch) return fail(MMX_E_INVALID, "mmx_adam_step_peer: null pointer");
    if (world < 1 || world > kMaxWorld || rank < 0 || rank >= world) return fail(MMX_E_INVALID, "mmx_adam_step_peer: rank %d / world %d (<= %d)", rank, world, kMaxWorld);
    if (n <= 0 || (n & 3)) return fail(MMX_E_INVALID, "mmx_adam_step_peer: the bucket length must be a positive multiple of 4 floats");
    if ((((uintptr_t)p) | ((uintptr_t)m) | ((uintptr_t)v)) & 15) return fail(MMX_E_INVALID, "mmx_adam_step_peer: buffers must be 16-byte aligned");
    PeerArgs a;
    a.p = p; a.m = m; a.v = v; a.peer_g = (const float* const*)peer_g; a.peer_flags = (unsigned int* const*)peer_flags; a.hp = hyper;
    a.epoch = epoch; a.abort_count = mmx_tc5_abort_ptr(); a.n = n; a.rank = rank; a.world = world;
    // two float4 per thread: K2 (30 K floats) 16 CTAs, K4 (183 K) 90 CTAs; fewer CTAs = fewer flags crossing NVLink
    long long want = ((n >> 2) + 2 * kPeerThreads - 1) / (2 * kPeerThreads);
    a.grid = (int)(want < 16 ? 16 : (want > kPeerCtas ? kPeerCtas : want));
    return launch_kernel(adam_peer_kernel, a.grid, kPeerThreads, 0, stream, kNoPdl, a);
}
#endif
