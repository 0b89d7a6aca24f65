// Launch layer shared by every translation unit of libmmx.so.
//
// nvcc build  -> motionmixerconv_b200/libmmx.so            (the product; CUDA only)
// g++ -DMMX_HOST_EMU -x c++ -> tests/emu/libmmx_emu.so     (test infrastructure: runs the very same
//                                                           kernel bodies phase by phase on the CPU)
#pragma once
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <mutex>

#include "../../include/mmx.h"
#include "mmx_common.cuh"

// defined in mmx_api_misc.cu: records the thread-local message returned by mmx_last_error()
int mmx_fail(int code, const char* fmt, ...);
#define fail mmx_fail
// address of the per-device counter of timed-out pipeline waits of the tcgen05 kernels (defined in mmx_api_mlp_tc5.cu)
int* mmx_tc5_abort_ptr();

namespace mmx {

// The library's only environment inputs are test hooks, read through env_int; each forces a plan so that a test can check it:
// MMX_MLP_V1 (generic MixerBlock kernels instead of the warp variant), MMX_CONV_S_FWD / MMX_CONV_S_BWD and
// MMX_CHEAD_S_FWD / MMX_CHEAD_S_BWD (ConvMixer half / head tile), MMX_CONV_X_GLOBAL (streamed-input ConvMixer backward),
// MMX_CHAN_STREAMED (tcgen05 channel-half plan), MMX_IO_NO_TC5 (fp32 embedding and output head kernels under tf32),
// MMX_CHEAD_EC (chunked ConvMixer head and its chunk width), MMX_ENC_HC (harmonic PoseEncoder forward: harmonics per chunk)
// and MMX_ENC_BWD_ROWS (harmonic PoseEncoder backward: staged frames).
static inline int env_int(const char* name, int dflt) {
    const char* s = getenv(name);
    return s && *s ? atoi(s) : dflt;
}

#if defined(MMX_HOST_EMU)
// ----------------------------------------------------------------------------- CPU emulator
struct DevInfo { int sms = 4; int max_smem = 227 * 1024; };
static inline DevInfo dev_info() { return DevInfo(); }

template <class Body, class Args, int OCC = 1>
static int launch(const Args& a, int grid, int block, size_t smem_bytes, void*) {
    std::vector<float> buf(smem_bytes / 4 + 8);
    float* sm = buf.data();
    while (((uintptr_t)sm) & 15) ++sm;
    for (int b = 0; b < grid; ++b) {
        for (size_t i = 0; i < smem_bytes / 4; ++i) sm[i] = NAN;   // poison: catches reads of unwritten smem
        Exec ex{block, b, grid, sm};
        Body::run(ex, a);
    }
    return MMX_OK;
}
#else
// ----------------------------------------------------------------------------- CUDA
struct DevInfo { int sms; int max_smem; };
static inline DevInfo dev_info() {
    static std::mutex mu;
    static DevInfo cache[64];
    static bool have[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) dev = 0;
    std::lock_guard<std::mutex> lk(mu);
    if (!have[dev]) {
        cudaDeviceGetAttribute(&cache[dev].sms, cudaDevAttrMultiProcessorCount, dev);
        cudaDeviceGetAttribute(&cache[dev].max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        have[dev] = true;
    }
    return cache[dev];
}

// values of launch_kernel's `pdl` argument
constexpr bool kPdl = true, kNoPdl = false;

// The one place a kernel of libmmx.so is launched.  Dynamic shared memory above 48 KB needs an opt-in per (kernel, device); with
// it, and on every programmatic dependent launch, ask for the full shared-memory carve-out: the planners size tiles so that two
// or more CTAs fit one SM, and otherwise the driver may pick an L1/shared split that holds fewer.
// pdl = kPdl (programmatic dependent launch): the kernel's parameter-only prologue may overlap the tail of the previous kernel in
// the stream.  Only for kernels that call griddepcontrol.wait before touching anything a predecessor writes (the tcgen05 family).
template <class K, class... A>
static int launch_kernel(K kern, dim3 grid, int block, size_t smem, void* stream, bool pdl, const A&... args) {
    const bool opt_in = smem > 48 * 1024;
    if (opt_in || pdl) {
        static std::mutex mu;
        static std::map<std::pair<const void*, int>, size_t> configured;     // (kernel, device) -> shared memory opted in to
        int dev = 0;
        cudaGetDevice(&dev);
        std::lock_guard<std::mutex> lk(mu);
        auto it = configured.find({(const void*)kern, dev});
        if (it == configured.end() || (opt_in && it->second < smem)) {
            if (opt_in) {
                cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                if (e != cudaSuccess) return fail(MMX_E_CUDA, "cudaFuncSetAttribute(%zu): %s", smem, cudaGetErrorString(e));
            }
            cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
            configured[{(const void*)kern, dev}] = opt_in ? smem : 0;
        }
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kern, args...);
    if (e != cudaSuccess) {
        cudaGetLastError();             // reported here: keep it from surfacing again at the caller's next error check
        return fail(MMX_E_CUDA, "kernel launch: %s", cudaGetErrorString(e));
    }
    return MMX_OK;
}

template <class Body, class Args>
static __global__ void __launch_bounds__(256) mmx_kernel(const Args a) {
    extern __shared__ float4 mmx_smem_raw[];
    Exec ex{(int)blockDim.x, (int)blockIdx.x, (int)gridDim.x, reinterpret_cast<float*>(mmx_smem_raw)};
    Body::run(ex, a);
}

// same kernel compiled for two resident CTAs per SM (<= 128 registers per thread)
template <class Body, class Args>
static __global__ void __launch_bounds__(256, 2) mmx_kernel_occ2(const Args a) {
    extern __shared__ float4 mmx_smem_raw[];
    Exec ex{(int)blockDim.x, (int)blockIdx.x, (int)gridDim.x, reinterpret_cast<float*>(mmx_smem_raw)};
    Body::run(ex, a);
}

template <class Body, class Args, int OCC = 1>
static int launch(const Args& a, int grid, int block, size_t smem_bytes, void* stream) {
    if constexpr (OCC >= 2) return launch_kernel(mmx_kernel_occ2<Body, Args>, grid, block, smem_bytes, stream, kNoPdl, a);
    else return launch_kernel(mmx_kernel<Body, Args>, grid, block, smem_bytes, stream, kNoPdl, a);
}
#endif

// Occupancy arithmetic.  Every resident CTA also takes 1 KB of the SM's shared memory that the kernel does not see, which is
// why an SM holds max_smem + 1 KB in all.
// CTAs of `smem` bytes of dynamic shared memory that fit on one SM, in [1, cap]
static inline int ctas_per_sm(const DevInfo& di, size_t smem, int cap) {
    return imax(1, imin(cap, (int)((di.max_smem + 1024) / (smem + 1024))));
}
// dynamic shared memory per CTA that leaves room for n CTAs per SM (and 1 KB of slack)
static inline int smem_budget(const DevInfo& di, int n) { return (di.max_smem + 1024) / n - 2048; }
// Tile search of the fp32 planners: the largest tile S in hi, hi - step, ... >= lo whose shared memory bytes_of(S) leaves room
// for two CTAs per SM, else the largest that fits one CTA; 0 if none fits.  two_cta_first = false: the one-CTA budget only.
template <class F>
static inline int fit_tile(const DevInfo& di, int hi, int lo, int step, bool two_cta_first, F bytes_of) {
    for (int pass = two_cta_first ? 0 : 1; pass < 2; ++pass) {
        const size_t budget = pass == 0 ? (size_t)smem_budget(di, 2) : (size_t)di.max_smem;
        for (int S = hi; S >= lo; S -= step)
            if ((size_t)bytes_of(S) <= budget) return S;
    }
    return 0;
}
// grid of ceil(work / per_cta) CTAs, in [1, k x SMs]
static inline int capped_grid(const DevInfo& di, long long work, long long per_cta, int k) {
    const long long want = (work + per_cta - 1) / per_cta, cap = (long long)di.sms * k;
    return (int)(want < 1 ? 1 : want < cap ? want : cap);
}

// grid for a persistent loop over `ntiles` tiles with at most `max_ctas` resident CTAs: balance the
// tiles so every CTA runs the same number of iterations (no ragged last wave)
static inline int balanced_grid(int ntiles, int max_ctas) {
    if (ntiles <= max_ctas) return ntiles > 0 ? ntiles : 1;
    const int waves = (ntiles + max_ctas - 1) / max_ctas;
    return (ntiles + waves - 1) / waves;
}
// grid for a persistent loop over n rows / sequences in tiles of S, each tile `bytes` of dynamic shared memory
static inline int tile_grid(const DevInfo& di, int n, int S, size_t bytes) {
    return balanced_grid((n + S - 1) / S, di.sms * ctas_per_sm(di, bytes, 8));
}

// Tile size in [lo, hi] (multiples of `step`) for a loop over n rows / sequences: CTAs are dealt round-robin to the SMs, so
// the makespan is (tiles on the busiest SM) x (tile size) -- e.g. 4096 sequences in tiles of 9 give 456 tiles = 4 rounds of
// 148 SMs at 9 sequences, tiles of 7 give 586 tiles = 4 rounds at 7.  Ties go to the larger tile (better weight reuse).
static inline int balanced_tile(int n, int hi, int lo, int step, int sms) {
    int best = hi;
    long long best_cost = -1;
    for (int S = hi; S >= imax(lo, 1); S -= step) {
        const int tiles = (n + S - 1) / S;
        const long long cost = (long long)((tiles + sms - 1) / sms) * S;
        if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = S; }
    }
    return best;
}

static inline Dropout make_dropout(const MmxDropout& s, int training) {
    Dropout d;
    d.seed_lo = (uint32_t)(s.seed & 0xffffffffull);
    d.seed_hi = (uint32_t)(s.seed >> 32);
    d.step = s.step;
    d.step_ptr = s.step_dev;
    if (training && s.p > 0.0f) {
        double t = (double)s.p * 4294967296.0;
        d.thresh = t >= 4294967295.0 ? 0xffffffffu : (uint32_t)(t + 0.5);
        if (d.thresh == 0u) d.thresh = 1u;
        d.scale = 1.0f / (1.0f - s.p);
    } else {
        d.thresh = 0u;
        d.scale = 1.0f;
    }
    return d;
}




constexpr int kThreads = 256;

// zero a device buffer on the stream (memset node: legal inside CUDA-graph capture)
static inline int zero_async(void* p, size_t bytes, void* stream) {
#if defined(MMX_HOST_EMU)
    (void)stream;
    memset(p, 0, bytes);
    return MMX_OK;
#else
    cudaError_t e = cudaMemsetAsync(p, 0, bytes, (cudaStream_t)stream);
    if (e != cudaSuccess) return fail(MMX_E_CUDA, "cudaMemsetAsync: %s", cudaGetErrorString(e));
    return MMX_OK;
#endif
}

}  // namespace mmx
