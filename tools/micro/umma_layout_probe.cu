// Layout discovery for tcgen05 shared-memory operands (SWIZZLE_NONE, kind::tf32): which shared-memory WORD does the tensor
// core read as element (mn, k) of an MN-major operand for a given (LBO, SBO)?  The operand region is filled with its own word
// index (two passes: low 11 bits / high bits, both exact in TF32), the other operand is a known-good K-major one-hot matrix.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O2 -o tools/micro/umma_layout_probe tools/micro/umma_layout_probe.cu
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "tc5_probe.cuh"
using namespace mmx::tc5;

constexpr int REGION_WORDS = 40 * 1024;   // 160 KB operand region under test

struct Cfg { int which; uint32_t lbo, sbo; int lt; };   // which: 0 = A is MN-major (B one-hot K-major), 1 = B is MN-major (A one-hot K-major)

__global__ void __launch_bounds__(128) probe(Cfg cfg, int pass, float* out /*[128][16]*/, int* abort_out) {
    extern __shared__ __align__(1024) uint8_t smem[];
    float* region = reinterpret_cast<float*>(smem);
    float* onehot = region + REGION_WORDS;                         // K-major one-hot [128 rows][8 k]: 2 panels x 2 KB
    uint64_t* bars = reinterpret_cast<uint64_t*>(onehot + 2 * 128 * 4);
    uint32_t* tslot = reinterpret_cast<uint32_t*>(bars + 2);
    volatile int* abortf = reinterpret_cast<volatile int*>(tslot + 1);
    const int tid = threadIdx.x, warp = tid >> 5;
    if (tid == 0) { mbar_init(&bars[0], 1); *abortf = 0; fence_mbar_init(); }
    if (warp == 0) tmem_alloc<32>(tslot);
    for (int w = tid; w < REGION_WORDS; w += 128) region[w] = (float)(pass == 0 ? (w & 0x7ff) : (w >> 11));
    for (int i = tid; i < 2 * 128 * 4; i += 128) {
        const int panel = i / (128 * 4), rr = (i / 4) % 128, cc = i % 4;
        onehot[i] = (rr == panel * 4 + cc) ? 1.0f : 0.0f;          // element (row rr, k) = (rr == k)
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tslot;
    if (tid == 0) {
        const uint64_t d_mn = smem_desc(smem_u32(region), cfg.lbo, cfg.sbo) | ((uint64_t)cfg.lt << 61);
        const uint64_t d_oh = desc_kmajor(smem_u32(onehot), 128 * 16, 0);
        if (cfg.which == 0) mma_ss(tmem, d_mn, d_oh, idesc_tf32(128, 16, 1, 0), 0);   // D[m][n] = A[m][k = n]
        else if (cfg.which == 1) mma_ss(tmem, d_oh, d_mn, idesc_tf32(128, 16, 0, 1), 0);   // D[m][n] = B[n][k = m]   (m < 8)
        else                mma_ss(tmem, d_mn, d_oh, idesc_tf32(128, 16, 0, 0), 0);   // sanity: A K-major with the given LBO/SBO
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
        {2, 2048, 128, 0},
        {0, 4096, 512, 1}, {0, 512, 4096, 1}, {0, 8192, 1024, 1}, {1, 4096, 512, 1}, {1, 512, 4096, 1},
        {0, 4096, 1024, 2}, {0, 1024, 4096, 2}, {1, 4096, 1024, 2},
    };
    float* dout; int* dab;
    cudaMalloc(&dout, 128 * 16 * 4); cudaMalloc(&dab, 4);
    const size_t smem = REGION_WORDS * 4 + 2 * 128 * 16 + 256;
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
        printf("=== %s MN-major, LBO %u SBO %u layout_type %d (abort %d): byte offset of element (mn, k)\n", c.which == 0 ? "A" : "B", c.lbo, c.sbo, c.lt, ab);
        printf("  raw pass0 row0: "); for (int k = 0; k < 16; ++k) printf("%g ", lo[k]); printf("| row1: "); for (int k = 0; k < 16; ++k) printf("%g ", lo[16 + k]); printf("\n");
        if (c.which != 1) {
            const int ms[] = {0, 1, 2, 3, 4, 5, 7, 8, 9, 12, 16, 32, 64, 127};
            for (int m : ms) {
                printf("  mn=%3d:", m);
                for (int k = 0; k < 8; ++k) printf(" %6d", 4 * ((int)lo[m * 16 + k] + 2048 * (int)hi[m * 16 + k]));
                printf("\n");
            }
        } else {
            const int ns[] = {0, 1, 2, 3, 4, 5, 7, 8, 9, 12, 15};
            for (int n : ns) {
                printf("  mn=%3d:", n);
                for (int k = 0; k < 8; ++k) printf(" %6d", 4 * ((int)lo[k * 16 + n] + 2048 * (int)hi[k * 16 + n]));
                printf("\n");
            }
        }
    }
    return 0;
}
