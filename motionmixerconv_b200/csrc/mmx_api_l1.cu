// Joint-angle training loss of the reference: mean over (sequence, frame) rows of the L1 distance over the angle dimensions,
//     loss = torch.mean(torch.sum(torch.abs(pred.reshape(-1, out_n, D) - gt), dim=2).view(-1))
// (h36m/train_mixer_h36m.py:187, train_autoreg_mixer_h36m.py:209-210), fused with its gradient like mmx_mpjpe_fwd_bwd.
#include "mmx_launch.cuh"

#if defined(MMX_HOST_EMU)
extern "C" int mmx_l1_fwd_bwd(const float*, const float*, float*, float*, long long, int, float, void*) {
    return fail(MMX_E_UNSUPPORTED, "mmx_l1_fwd_bwd: not in the emulator");
}
#else
using namespace mmx;

namespace {
// *loss_sum += sum |pred - gt| ; dpred = gscale * sign(pred - gt) / rows   (sign(0) = 0, as torch.abs' backward)
__global__ void __launch_bounds__(256) l1_kernel(const float* __restrict__ pred, const float* __restrict__ gt, float* __restrict__ dpred,
                                                 float* loss_sum, long long n, float g) {
    float acc = 0.0f;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float d = pred[i] - gt[i];
        acc += fabsf(d);
        if (dpred) dpred[i] = d > 0.0f ? g : (d < 0.0f ? -g : 0.0f);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    __shared__ float part[8];
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0.0f;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += part[w];
        atomicAdd(loss_sum, s);
    }
}
}  // namespace

extern "C" int mmx_l1_fwd_bwd(const float* pred, const float* gt, float* dpred, float* loss_sum, long long rows, int D, float gscale, void* stream) {
    if (!pred || !gt || !loss_sum) return fail(MMX_E_INVALID, "mmx_l1_fwd_bwd: null tensor");
    if (rows <= 0 || D <= 0) return fail(MMX_E_INVALID, "mmx_l1_fwd_bwd: bad sizes");
    const long long n = rows * D;
    return launch_kernel(l1_kernel, capped_grid(dev_info(), n, 1024, 4), 256, 0, stream, kNoPdl, pred, gt, dpred, loss_sum, n, gscale / (float)rows);
}
#endif
