// Launch helper of the tcgen05 kernel families (MixerBlock halves, linear layer, output head).
#pragma once
#include <mutex>

#include "mmx_launch.cuh"

// address of the per-device counter of timed-out pipeline waits (defined in mmx_api_mlp_tc5.cu)
int* mmx_tc5_abort_ptr();

namespace mmx {

template <class K, class... A>
static int launch_tc5v(K kern, int grid, int block, size_t smem, void* stream, const A&... a) {
    struct Conf { const void* fn; int dev; size_t smem; };
    static Conf conf[128];
    static int nconf = 0;
    static std::mutex mu;
    int dev = 0;
    cudaGetDevice(&dev);
    {
        std::lock_guard<std::mutex> lk(mu);
        int slot = -1;
        for (int i = 0; i < nconf; ++i)
            if (conf[i].fn == (const void*)kern && conf[i].dev == dev) slot = i;
        if (slot < 0 || conf[slot].smem < smem) {
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return fail(MMX_E_CUDA, "cudaFuncSetAttribute(%zu): %s", smem, cudaGetErrorString(e));
            cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
            if (slot < 0 && nconf < 128) slot = nconf++;
            if (slot >= 0) conf[slot] = Conf{(const void*)kern, dev, smem};
        }
    }
    // programmatic dependent launch: the kernel's parameter-only prologue may overlap the tail of the previous kernel in the
    // stream (every kernel of this family calls griddepcontrol.wait before touching anything a predecessor writes)
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kern, a...);
    if (e != cudaSuccess) return fail(MMX_E_CUDA, "kernel launch: %s", cudaGetErrorString(e));
    return MMX_OK;
}
template <class K, class A>
static int launch_tc5(K kern, const A& a, int grid, int block, size_t smem, void* stream) {
    return launch_tc5v(kern, grid, block, smem, stream, a);
}

}  // namespace mmx
