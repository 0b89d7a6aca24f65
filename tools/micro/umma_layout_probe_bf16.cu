// Layout discovery for tcgen05 kind::f16 (bf16) shared-memory operands, SWIZZLE_NONE: which 2-byte ELEMENT does the tensor core
// read as element (mn, k) of a K-major / MN-major operand for a given (LBO, SBO)?  The operand region is filled with its own
// element index (two passes of 8 bits, exact in bf16); the other operand is a K-major one-hot matrix.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O2 -o tools/micro/umma_layout_probe_bf16 tools/micro/umma_layout_probe_bf16.cu
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <cuda_bf16.h>

#include "tc5_probe.cuh"
using namespace mmx::tc5;

constexpr int REGION_ELEMS = 64 * 1024;   // 128 KB operand region under test

struct Cfg { int which; uint32_t lbo, sbo; };   // 0: A MN-major, 1: B MN-major, 2: A K-major (sanity)

__global__ void __launch_bounds__(128) probe(Cfg cfg, int pass, float* out /*[128][16]*/, int* abort_out) {
    extern __shared__ __align__(1024) uint8_t smem[];
    __nv_bfloat16* region = reinterpret_cast<__nv_bfloat16*>(smem);
    __nv_bfloat16* onehot = region + REGION_ELEMS;                  // K-major one-hot [128 rows][16 k]: 2 panels x (128 rows x 16 B)
    uint64_t* bars = reinterpret_cast<uint64_t*>(onehot + 2 * 128 * 8);
    uint32_t* tslot = reinterpret_cast<uint32_t*>(bars + 2);
    volatile int* abortf = reinterpret_cast<volatile int*>(tslot + 1);
    const int tid = threadIdx.x, warp = tid >> 5;
    if (tid == 0) { mbar_init(&bars[0], 1); *abortf = 0; fence_mbar_init(); }
    if (warp == 0) tmem_alloc<32>(tslot);
    for (int w = tid; w < REGION_ELEMS; w += 128) region[w] = __float2bfloat16((float)(pass == 0 ? (w & 0xff) : (w >> 8)));
    for (int i = tid; i < 2 * 128 * 8; i += 128) {
        const int panel = i / (128 * 8), rr = (i / 8) % 128, cc = i % 8;
        onehot[i] = __float2bfloat16((rr == panel * 8 + cc) ? 1.0f : 0.0f);   // element (row rr, k) = (rr == k), k < 16
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tslot;
    if (tid == 0) {
        const uint64_t d_x = smem_desc(smem_u32(region), cfg.lbo, cfg.sbo);
        const uint64_t d_oh = smem_desc(smem_u32(onehot), 128 * 16, 128);
        if (cfg.which == 0) mma_f16(tmem, d_x, d_oh, idesc_bf16(128, 16, 1, 0), 0);        // D[m][n] = A[m][k = n]
        else if (cfg.which == 1) mma_f16(tmem, d_oh, d_x, idesc_bf16(128, 16, 0, 1), 0);   // D[m][n] = B[n][k = m]   (m < 16)
        else mma_f16(tmem, d_x, d_oh, idesc_bf16(128, 16, 0, 0), 0);                      // sanity: A K-major
        mma_commit(&bars[0]);
    }
    mbar_wait(&bars[0], 0, abortf);
    tc_fence_after();
    float v[16];
    tmem_ld16(tmem_addr(tmem, warp, 0), v);
    tmem_wait_ld();
    for (int j = 0; j < 16; ++j) out[tid * 16 + j] = v[j];
    if (tid == 0) *abort_out = *abortf;
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<32>(tmem);
}

int main() {
    const Cfg cfgs[] = {
        {2, 2048, 128},
        {0, 128, 2048}, {0, 2048, 128}, {0, 256, 4096},
        {1, 128, 2048}, {1, 2048, 128}, {1, 256, 4096},
    };
    float* dout; int* dab;
    cudaMalloc(&dout, 128 * 16 * 4); cudaMalloc(&dab, 4);
    const size_t smem = REGION_ELEMS * 2 + 2 * 128 * 16 + 256;
    cudaFuncSetAttribute(probe, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    std::vector<float> lo(128 * 16), hi(128 * 16);
    for (const Cfg& c : cfgs) {
        int ab = 0;
        for (int pass = 0; pass < 2; ++pass) {
            probe<<<1, 128, smem>>>(c, pass, dout, dab);
            cudaError_t e = cudaDeviceSynchronize();
            if (e != cudaSuccess) { printf("kernel error: %s\n", cudaGetErrorString(e)); return 2; }
            cudaMemcpy(pass == 0 ? lo.data() : hi.data(), dout, 128 * 16 * 4, cudaMemcpyDeviceToHost);
            cudaMemcpy(&ab, dab, 4, cudaMemcpyDeviceToHost);
        }
        printf("=== bf16 %s, LBO %u SBO %u (abort %d): BYTE offset of element (mn, k), k = 0..15\n",
               c.which == 0 ? "A MN-major" : c.which == 1 ? "B MN-major" : "A K-major", c.lbo, c.sbo, ab);
        if (c.which != 1) {
            const int ms[] = {0, 1, 2, 3, 7, 8, 9, 15, 16, 17, 32, 64, 127};
            for (int m : ms) {
                printf("  mn=%3d:", m);
                for (int k = 0; k < 16; ++k) printf(" %6d", 2 * ((int)lo[m * 16 + k] + 256 * (int)hi[m * 16 + k]));
                printf("\n");
            }
        } else {
            const int ns[] = {0, 1, 2, 3, 7, 8, 9, 15};
            for (int n : ns) {
                printf("  mn=%3d:", n);
                for (int k = 0; k < 16; ++k) printf(" %6d", 2 * ((int)lo[k * 16 + n] + 256 * (int)hi[k * 16 + n]));
                printf("\n");
            }
        }
    }
    return 0;
}
