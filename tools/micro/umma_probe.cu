// tcgen05 / TMEM / bulk-copy probe (sm_100a): checks, against a CPU product of exactly representable inputs, every operand
// form the MixerBlock channel-half kernels rely on (mmx_tc5.cuh panel layout):
//   T1  D = A * B^T        A K-major smem, B K-major smem         (forward GEMMs)
//   T2  D = A * B^T        A from TMEM (tcgen05.st), B K-major    (the "lo" operand path)
//   T3  D = X^T * Y        A MN-major smem, B MN-major smem       (weight gradients, K = rows)
//   T4  D = A * W          A K-major smem, B MN-major smem        (data gradients with the untransposed weight)
//   T5  accumulate flag (T1 issued twice), T6 rounding of fp32 words fed to kind::tf32, bulk copy in/out.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O2 -o tools/micro/umma_probe tools/micro/umma_probe.cu
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "tc5_probe.cuh"

using namespace mmx::tc5;

constexpr int R = 128;            // rows of the activation tiles
constexpr int KP = 56;            // padded contraction width of T1/T2/T4
constexpr int N1 = 64;            // output width
constexpr int AP_COLS = 128;      // A buffer is allocated with 32 panels so that T3 (M = 128 columns) stays inside it
constexpr uint32_t PANEL_A = R * 16, PANEL_B = 64 * 16;

struct Out {
    float d1[R * N1], d2[R * N1], d3[128 * N1], d4[R * N1], d5[R * N1], d6[R * 16];
    float bulk_echo[R * 16];
    int abort_flag, tmem_base;
};

__global__ void __launch_bounds__(128) probe(const float* __restrict__ a_img, const float* __restrict__ b_img, const float* __restrict__ y_img,
                                             const float* __restrict__ w_img, const float* __restrict__ a_rows, Out* out) {
    extern __shared__ __align__(1024) uint8_t smem[];
    float* sA = reinterpret_cast<float*>(smem);                         // 32 panels x 2 KB = 64 KB
    float* sY = sA + 32 * R * 4;                                        // 16 panels x 2 KB = 32 KB  ([128 rows][64 cols])
    float* sB = sY + 16 * R * 4;                                        // 14 panels x 1 KB          ([64 rows][56 cols])
    float* sW = sB + 14 * 64 * 4;                                       // 16 panels x 1 KB          ([64 rows = k][64 cols = n])
    uint64_t* bars = reinterpret_cast<uint64_t*>(sW + 16 * 64 * 4);     // [0] bulk, [1] mma
    uint32_t* tslot = reinterpret_cast<uint32_t*>(bars + 4);
    volatile int* abortf = reinterpret_cast<volatile int*>(tslot + 1);
    const int tid = threadIdx.x, warp = tid >> 5;

    if (tid == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        *abortf = 0;
        fence_mbar_init();
    }
    if (warp == 0) tmem_alloc<512>(tslot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tslot;

    // ---- bulk copy global -> shared of the A image (64 KB, two copies), everything else by plain loads
    if (tid == 0) {
        mbar_expect_tx(&bars[0], 32 * PANEL_A);
        bulk_g2s(sA, a_img, 16 * PANEL_A, &bars[0]);
        bulk_g2s(sA + 16 * R * 4, a_img + 16 * R * 4, 16 * PANEL_A, &bars[0]);
    }
    for (int i = tid; i < 16 * R * 4; i += 128) sY[i] = y_img[i];
    for (int i = tid; i < 14 * 64 * 4; i += 128) sB[i] = b_img[i];
    for (int i = tid; i < 16 * 64 * 4; i += 128) sW[i] = w_img[i];
    mbar_wait(&bars[0], 0, abortf);
    // A rows into TMEM columns [256, 256+56) for T2 (thread = row)
    for (int c = 0; c < KP; c += 4) {
        const float* p = a_rows + tid * KP + c;
        tmem_st4(tmem_addr(tmem, warp, 256 + c), p[0], p[1], p[2], p[3]);
    }
    tmem_wait_st();
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    uint32_t phase = 0;
    const uint32_t aB = smem_u32(sA), yB = smem_u32(sY), bB = smem_u32(sB), wB = smem_u32(sW);
    if (tid == 0) {
        // T1: cols 0..63
        for (int k = 0; k < KP; k += 8)
            mma_ss(tmem + 0, desc_kmajor(aB, PANEL_A, k), desc_kmajor(bB, PANEL_B, k), idesc_tf32(128, N1, 0, 0), k > 0);
        // T2: cols 64..127, A from TMEM
        for (int k = 0; k < KP; k += 8)
            mma_ts(tmem + 64, tmem + 256 + k, desc_kmajor(bB, PANEL_B, k), idesc_tf32(128, N1, 0, 0), k > 0);
        // T3: cols 128..191: D[m][n] = sum_r A[r][m] * Y[r][n]
        for (int r = 0; r < R; r += 8)
            mma_ss(tmem + 128, desc_mnmajor(aB, PANEL_A, r, 0), desc_mnmajor(yB, PANEL_A, r, 0), idesc_tf32(128, N1, 1, 1), r > 0);
        // T4: cols 192..255: D[r][n] = sum_k A[r][k] * W[k][n]
        for (int k = 0; k < KP; k += 8)
            mma_ss(tmem + 192, desc_kmajor(aB, PANEL_A, k), desc_mnmajor(wB, PANEL_B, k, 0), idesc_tf32(128, N1, 0, 1), k > 0);
        // T5: cols 320..383: T1 twice with the accumulate flag
        for (int rep = 0; rep < 2; ++rep)
            for (int k = 0; k < KP; k += 8)
                mma_ss(tmem + 320, desc_kmajor(aB, PANEL_A, k), desc_kmajor(bB, PANEL_B, k), idesc_tf32(128, N1, 0, 0), (rep | k) > 0);
        mma_commit(&bars[1]);
    }
    mbar_wait(&bars[1], phase, abortf);
    phase ^= 1;
    tc_fence_after();
    for (int c = 0; c < N1; c += 8) {
        float v[8];
        tmem_ld8(tmem_addr(tmem, warp, 0 + c), v);   tmem_wait_ld();
        for (int j = 0; j < 8; ++j) out->d1[tid * N1 + c + j] = v[j];
        tmem_ld8(tmem_addr(tmem, warp, 64 + c), v);  tmem_wait_ld();
        for (int j = 0; j < 8; ++j) out->d2[tid * N1 + c + j] = v[j];
        tmem_ld8(tmem_addr(tmem, warp, 128 + c), v); tmem_wait_ld();
        for (int j = 0; j < 8; ++j) out->d3[tid * N1 + c + j] = v[j];
        tmem_ld8(tmem_addr(tmem, warp, 192 + c), v); tmem_wait_ld();
        for (int j = 0; j < 8; ++j) out->d4[tid * N1 + c + j] = v[j];
        tmem_ld8(tmem_addr(tmem, warp, 320 + c), v); tmem_wait_ld();
        for (int j = 0; j < 8; ++j) out->d5[tid * N1 + c + j] = v[j];
    }
    // T6: how are fp32 words with low mantissa bits treated?  panel 0 of sA := per-row test values, B := identity-ish
    tc_fence_before();
    __syncthreads();
    {
        // A[r][0..3] = (1 + 2^-11 + 2^-13, 1 + 2^-11, 1 + 2^-10 + 2^-11, 1 + 2^-12) ; other K columns zero
        const float t0 = 1.0f + 0x1p-11f + 0x1p-13f, t1 = 1.0f + 0x1p-11f, t2 = 1.0f + 0x1p-10f + 0x1p-11f, t3 = 1.0f + 0x1p-12f;
        float* p0 = sA + tid * 4;
        p0[0] = t0; p0[1] = t1; p0[2] = t2; p0[3] = t3;
        float* p1 = sA + R * 4 + tid * 4;
        p1[0] = p1[1] = p1[2] = p1[3] = 0.0f;
        // B [16 rows = n][8 cols = k]: B[n][k] = (n == k)
        for (int i = tid; i < 2 * 64 * 4; i += 128) {
            const int panel = i / (64 * 4), rr = (i / 4) % 64, cc = i % 4;
            sB[i] = (rr == panel * 4 + cc) ? 1.0f : 0.0f;
        }
    }
    fence_async_smem();
    __syncthreads();
    tc_fence_after();
    if (tid == 0) {
        mma_ss(tmem + 384, desc_kmajor(aB, PANEL_A, 0), desc_kmajor(bB, PANEL_B, 0), idesc_tf32(128, 16, 0, 0), 0);
        mma_commit(&bars[1]);
    }
    mbar_wait(&bars[1], phase, abortf);
    phase ^= 1;
    tc_fence_after();
    {
        float v[16];
        tmem_ld16(tmem_addr(tmem, warp, 384), v);
        tmem_wait_ld();
        for (int j = 0; j < 16; ++j) out->d6[tid * 16 + j] = v[j];
    }
    // bulk store shared -> global of panel 0 of sA
    __syncthreads();
    if (tid == 0) {
        fence_async_smem();
        bulk_s2g(out->bulk_echo, sA, PANEL_A);
        bulk_commit();
        bulk_wait_all0();
        out->abort_flag = *abortf;
        out->tmem_base = (int)tmem;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<512>(tmem);
}

static void to_panels(const std::vector<float>& m, int rows, int cols, int alloc_rows, int alloc_cols, std::vector<float>& img) {
    img.assign((size_t)(alloc_cols / 4) * alloc_rows * 4, 0.0f);
    for (int r = 0; r < rows; ++r)
        for (int c = 0; c < cols; ++c) img[(size_t)(c / 4) * alloc_rows * 4 + r * 4 + (c % 4)] = m[(size_t)r * cols + c];
}

static int cmp(const char* name, const float* got, const std::vector<float>& want, int n) {
    int bad = 0;
    double maxd = 0;
    for (int i = 0; i < n; ++i) {
        double d = fabs((double)got[i] - want[i]);
        if (d > maxd) maxd = d;
        if (d > 1e-6 * (1 + fabs(want[i]))) ++bad;
    }
    printf("%-28s %s  mismatches %d / %d  max|diff| %.3g\n", name, bad ? "FAIL" : "ok  ", bad, n, maxd);
    return bad != 0;
}

int main() {
    srand(7);
    auto rnd = [](int lim) { return (float)((rand() % (2 * lim + 1)) - lim); };
    std::vector<float> A((size_t)R * AP_COLS), B((size_t)N1 * KP), Y((size_t)R * N1), W((size_t)64 * N1, 0.0f), Arows((size_t)R * KP);
    for (auto& v : A) v = rnd(4);
    for (auto& v : B) v = rnd(3);
    for (auto& v : Y) v = rnd(3);
    for (int k = 0; k < KP; ++k)
        for (int n = 0; n < N1; ++n) W[(size_t)k * N1 + n] = rnd(3);
    for (int r = 0; r < R; ++r)
        for (int k = 0; k < KP; ++k) Arows[(size_t)r * KP + k] = A[(size_t)r * AP_COLS + k];
    std::vector<float> aimg, bimg, yimg, wimg;
    to_panels(A, R, AP_COLS, R, AP_COLS, aimg);
    to_panels(B, N1, KP, 64, KP, bimg);
    to_panels(Y, R, N1, R, N1, yimg);
    to_panels(W, 64, N1, 64, N1, wimg);

    std::vector<float> w1((size_t)R * N1), w3((size_t)128 * N1), w4((size_t)R * N1), w5((size_t)R * N1);
    for (int r = 0; r < R; ++r)
        for (int n = 0; n < N1; ++n) {
            double s = 0, s4 = 0;
            for (int k = 0; k < KP; ++k) { s += (double)A[(size_t)r * AP_COLS + k] * B[(size_t)n * KP + k]; s4 += (double)A[(size_t)r * AP_COLS + k] * W[(size_t)k * N1 + n]; }
            w1[(size_t)r * N1 + n] = (float)s; w5[(size_t)r * N1 + n] = (float)(2 * s); w4[(size_t)r * N1 + n] = (float)s4;
        }
    for (int m = 0; m < 128; ++m)
        for (int n = 0; n < N1; ++n) {
            double s = 0;
            for (int r = 0; r < R; ++r) s += (double)A[(size_t)r * AP_COLS + m] * Y[(size_t)r * N1 + n];
            w3[(size_t)m * N1 + n] = (float)s;
        }

    float *da, *db, *dy, *dw, *dar;
    Out* dout;
    cudaMalloc(&da, aimg.size() * 4); cudaMalloc(&db, bimg.size() * 4); cudaMalloc(&dy, yimg.size() * 4);
    cudaMalloc(&dw, wimg.size() * 4); cudaMalloc(&dar, Arows.size() * 4); cudaMalloc(&dout, sizeof(Out));
    cudaMemcpy(da, aimg.data(), aimg.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(db, bimg.data(), bimg.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dy, yimg.data(), yimg.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dw, wimg.data(), wimg.size() * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dar, Arows.data(), Arows.size() * 4, cudaMemcpyHostToDevice);
    cudaMemset(dout, 0xff, sizeof(Out));
    const size_t smem = (32 * R * 4 + 16 * R * 4 + 14 * 64 * 4 + 16 * 64 * 4) * 4 + 256;
    cudaFuncSetAttribute(probe, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    probe<<<1, 128, smem>>>(da, db, dy, dw, dar, dout);
    cudaError_t e = cudaDeviceSynchronize();
    printf("kernel: %s\n", cudaGetErrorString(e));
    if (e != cudaSuccess) return 2;
    Out* h = (Out*)malloc(sizeof(Out));
    cudaMemcpy(h, dout, sizeof(Out), cudaMemcpyDeviceToHost);
    printf("abort_flag %d tmem_base 0x%x\n", h->abort_flag, h->tmem_base);
    int bad = 0;
    bad += cmp("T1 SS K-major x K-major", h->d1, w1, R * N1);
    bad += cmp("T2 TS (A in TMEM)", h->d2, w1, R * N1);
    bad += cmp("T3 SS MN-major x MN-major", h->d3, w3, 128 * N1);
    bad += cmp("T4 SS K-major x MN-major", h->d4, w4, R * N1);
    bad += cmp("T5 accumulate", h->d5, w5, R * N1);
    printf("T6 tf32 conversion of fp32 words (row 0): in = 1+2^-11+2^-13, 1+2^-11, 1+2^-10+2^-11, 1+2^-12\n   out-1 (units of 2^-10): ");
    for (int j = 0; j < 4; ++j) printf("%g ", (h->d6[j] - 1.0f) * 1024.0f);
    printf(" | cols 4..7: %g %g %g %g\n", h->d6[4], h->d6[5], h->d6[6], h->d6[7]);
    int be = 0;
    for (int r = 0; r < R; ++r) {
        const float want[4] = {1.0f + 0x1p-11f + 0x1p-13f, 1.0f + 0x1p-11f, 1.0f + 0x1p-10f + 0x1p-11f, 1.0f + 0x1p-12f};
        for (int j = 0; j < 4; ++j) be += h->bulk_echo[r * 4 + j] != want[j];
    }
    printf("bulk store echo              %s\n", be ? "FAIL" : "ok  ");
    bad += be != 0;
    printf(bad ? "PROBE FAILED\n" : "PROBE OK\n");
    return bad ? 1 : 0;
}
