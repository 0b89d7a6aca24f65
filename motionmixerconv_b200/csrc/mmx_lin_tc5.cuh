// Row-wise linear layer on the Blackwell tensor cores (tcgen05 + TMEM + bulk-copy engine), sm_100a:
//
//     y[r, :] = W x[r, :] + b          W: [N, K] (nn.Linear layout), rows r = 0 .. R-1
//
// Serves MlpMixer.conv (Conv2d(1,H,(1,D)) == per-frame Linear D -> H, h36m/mlp_mixer.py:268,325-327) and fc_out (Linear H -> D,
// mlp_mixer.py:300,335) in the reduced-precision mode, with the bf16x3 toolkit of mmx_tc5.cuh: 128-row tiles, one thread per
// (row, chunk set), bf16 hi+lo split operands in the 16-bit panel layout (one copy, both orientations), three MMAs per
// product, accumulators in TMEM.  Backward: dW = dY^T X (+ db from a ones column of X) accumulates in TMEM across the CTA's
// persistent loop and is flushed once; dx = dY W (optional) uses the untransposed weight as an MN-major operand.
#pragma once
#include "mmx_tc5.cuh"

namespace mmx {
namespace lin {

using namespace tc5;

struct LinArgs {
    const float* x;      // [R, K]
    const float* dy;     // backward: [R, N]
    float* out;          // forward: y [R, N]; backward: dx [R, K] (nullable)
    const float *w, *b;  // [N, K], [N]
    float *g_w, *g_b;    // backward, accumulated
    long long R;
    int K, N;
    int* abort_count;
};

// shared-memory layout (byte offsets from the 1024-aligned base; total includes the alignment slack).  KP: padded width of
// BOTH operand buffers (multiple of 16, > K so that column K can carry the ones of the bias gradient, >= N)
struct LinSmem {
    uint32_t x, y, w, sx, sy, bias, bars, total;
};
template <int KP>
MMX_HD LinSmem lin_smem(int K, int N, bool bwd) {
    using P = Panels<KP>;
    const uint32_t sx = up128(128u * K * 4u + 64u), sy = up128(128u * N * 4u + 64u);
    const uint32_t bx = umax(P::BUF, umax(sx, sy));               // X doubles as the staging tile of the output
    LinSmem m;
    uint32_t o = 0;
    m.x = o; o += bx;
    m.y = o; o += bwd ? bx : 0;                                     // backward: operand dY
    m.w = o; o += P::WBUF;
    m.sx = o; o += sx;                                              // x tile
    m.sy = o; o += bwd ? sy : 0;                                    // backward: dy tile
    m.bias = o; o += KP * 4;
    m.bars = o; o += 64 * 4;                                        // barriers, TMEM slot, abort flag
    m.total = o + 1024;
    return m;
}

// ------------------------------------------------------------------------------------------ forward
template <int KP, int VEC>
__global__ void __launch_bounds__(kCtaThreads) lin_fwd_kernel(const LinArgs a) {
    using P = Panels<KP>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int K = a.K, N = a.N;
    const LinSmem m = lin_smem<KP>(K, N, false);
    uint8_t* bufX = sm + m.x;                                 // operand X, later the output staging tile
    uint8_t* wb = sm + m.w;
    float* S = reinterpret_cast<float*>(sm + m.sx);
    float* bias = reinterpret_cast<float*>(sm + m.bias);
    uint64_t* bars = reinterpret_cast<uint64_t*>(sm + m.bars);
    uint32_t* tslot = reinterpret_cast<uint32_t*>(bars + 4);
    volatile int* abortf = reinterpret_cast<volatile int*>(tslot + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, qtr = warp & 3, half = warp >> 2;
    const int prow = qtr * 32 + lane;
    constexpr int TM_COLS = KP <= 64 ? 64 : 128;
    constexpr int NCH = KP / 8;
    cta_begin<TM_COLS>(bars, 2, abortf, tslot, tid);
    pdl_launch_dependents();
    for (int i = tid; i < (int)(P::WBUF / 16); i += kCtaThreads) reinterpret_cast<uint4*>(wb)[i] = make_uint4(0, 0, 0, 0);
    for (int c = tid; c < KP; c += kCtaThreads) bias[c] = c < N ? a.b[c] : 0.0f;
    __syncthreads();
    stage_weight<KP>(wb, a.w, N, K, nullptr, tid);
    pdl_wait();
    const long long ntiles = (a.R + 127) / 128;
    auto tile_rows = [&](long long t) { return (int)min((long long)128, a.R - t * 128); };
    if (warp == 0 && (long long)blockIdx.x < ntiles)
        stage_in<VEC>(S, a.x, (size_t)blockIdx.x * 128, tile_rows(blockIdx.x), K, K, &bars[0], lane);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tslot;
    const uint32_t xB = smem_u32(bufX), wB = smem_u32(wb);
    uint32_t ph_in = 0, ph_mma = 0;
    const int nchK = (K + 7) >> 3, nchN = (N + 7) >> 3;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int nrows = tile_rows(tile);
        const bool valid = prow < nrows;
        const float* srow = S + (size_t)prow * K;
        mbar_wait(&bars[0], ph_in, abortf);
        ph_in ^= 1;
        if (warp == 0) bulk_wait_read0();              // previous output (staged in the X region) has left shared memory
        __syncthreads();
#pragma unroll 1
        for (int c8 = half; c8 < NCH; c8 += kHalves) {
            float v[8];
            ld8<VEC>(srow, 8 * c8, (valid && c8 < nchK) ? K : 0, v);
            put_chunk(bufX, P::PLANE, P::PS, prow, c8, v);
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (warp == 0) {
            const long long next = tile + gridDim.x;
            if (next < ntiles) stage_in<VEC>(S, a.x, (size_t)next * 128, tile_rows(next), K, K, &bars[0], lane);
        }
        if (tid == 0) {
            tc_fence_after();
            gemm3<0, 0>(tmem, xB, xB + P::PLANE, P::PS, wB, wB + P::WPLANE, P::WPS, KP, KP / 16, false);
            mma_commit(&bars[1]);
        }
        mbar_wait(&bars[1], ph_mma, abortf);
        ph_mma ^= 1;
        tc_fence_after();
        {
            float* orow = reinterpret_cast<float*>(bufX) + (size_t)prow * N;
#pragma unroll 1
            for (int c8 = half; c8 < nchN; c8 += kHalves) {
                float u[8], b[8];
                tmem_ld8(tmem_addr(tmem, qtr, 8 * c8), u);
                ld8s(bias + 8 * c8, b);
                tmem_wait_ld();
#pragma unroll
                for (int j = 0; j < 8; ++j) u[j] += b[j];
                if (valid) st8<2>(orow, 8 * c8, N, u);
            }
        }
        tc_fence_before();
        fence_async_smem();
        __syncthreads();
        if (warp == 0) {
            if (lane == 0) bulk_s2g(a.out + (size_t)tile * 128 * N, bufX, (uint32_t)nrows * N * 4u);
            bulk_commit();
        }
    }
    cta_end<TM_COLS>(abortf, a.abort_count, tmem, tid);
}

// ------------------------------------------------------------------------------------------ backward
template <int KP, int VEC>
__global__ void __launch_bounds__(kCtaThreads) lin_bwd_kernel(const LinArgs a) {
    using P = Panels<KP>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int K = a.K, N = a.N;
    const bool want_dx = a.out != nullptr;
    const LinSmem m = lin_smem<KP>(K, N, true);
    uint8_t* bufX = sm + m.x;                                 // operand X (+ ones column at K), later the dx staging tile
    uint8_t* bufY = sm + m.y;                                 // operand dY
    uint8_t* wb = sm + m.w;
    float* SX = reinterpret_cast<float*>(sm + m.sx);
    float* SY = reinterpret_cast<float*>(sm + m.sy);
    uint64_t* bars = reinterpret_cast<uint64_t*>(sm + m.bars);
    uint32_t* tslot = reinterpret_cast<uint32_t*>(bars + 4);
    volatile int* abortf = reinterpret_cast<volatile int*>(tslot + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, qtr = warp & 3, half = warp >> 2;
    const int prow = qtr * 32 + lane;
    constexpr int TM_COLS = 2 * KP <= 128 ? 128 : 256;
    constexpr int NCH = KP / 8;
    cta_begin<TM_COLS>(bars, 2, abortf, tslot, tid);
    pdl_launch_dependents();
    for (int i = tid; i < (int)(P::WBUF / 16); i += kCtaThreads) reinterpret_cast<uint4*>(wb)[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();
    if (want_dx) stage_weight<KP>(wb, a.w, N, K, nullptr, tid);
    pdl_wait();
    const long long ntiles = (a.R + 127) / 128;
    auto tile_rows = [&](long long t) { return (int)min((long long)128, a.R - t * 128); };
    auto load_tile = [&](long long t) {
        const int nr = tile_rows(t);
        if (lane == 0) mbar_expect_tx(&bars[0], (uint32_t)nr * (K + N) * 4u);
        __syncwarp();
        if (lane == 0) {
            bulk_g2s(SX, a.x + (size_t)t * 128 * K, (uint32_t)nr * K * 4u, &bars[0]);
            bulk_g2s(SY, a.dy + (size_t)t * 128 * N, (uint32_t)nr * N * 4u, &bars[0]);
        }
    };
    if (warp == 0 && (long long)blockIdx.x < ntiles) load_tile(blockIdx.x);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tslot;
    const uint32_t tDW = tmem, tDX = tmem + KP;
    const uint32_t xB = smem_u32(bufX), yB = smem_u32(bufY), wB = smem_u32(wb);
    uint32_t ph_in = 0, ph_mma = 0;
    bool first = true;
    const int nchK = (K + 7) >> 3, nchN = (N + 7) >> 3;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int nrows = tile_rows(tile);
        const bool valid = prow < nrows;
        mbar_wait(&bars[0], ph_in, abortf);
        ph_in ^= 1;
        if (warp == 0) bulk_wait_read0();
        __syncthreads();
        const float* xrow = SX + (size_t)prow * K;
        const float* yrow = SY + (size_t)prow * N;
#pragma unroll 1
        for (int c8 = half; c8 < NCH; c8 += kHalves) {
            float v[8];
            ld8<VEC>(xrow, 8 * c8, (valid && c8 < nchK) ? K : 0, v);
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (valid && 8 * c8 + j == K) v[j] = 1.0f;          // ones column: dW[:, K] = db
            put_chunk(bufX, P::PLANE, P::PS, prow, c8, v);
            ld8<2>(yrow, 8 * c8, (valid && c8 < nchN) ? N : 0, v);
            put_chunk(bufY, P::PLANE, P::PS, prow, c8, v);
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (warp == 0) {
            const long long next = tile + gridDim.x;
            if (next < ntiles) load_tile(next);
        }
        if (tid == 0) {
            tc_fence_after();
            // dW[n][k] += sum_r dY[r][n] X[r][k]   (both MN-major, K = the 128 rows)
            gemm3<1, 1>(tDW, yB, yB + P::PLANE, P::PS, xB, xB + P::PLANE, P::PS, KP, 128 / 16, !first);
            // dx[r][k] = sum_n dY[r][n] W[n][k]    (A = dY K-major, B = W [N rows][K cols] read MN-major)
            if (want_dx) gemm3<0, 1>(tDX, yB, yB + P::PLANE, P::PS, wB, wB + P::WPLANE, P::WPS, KP, KP / 16, false);
            mma_commit(&bars[1]);
        }
        first = false;
        mbar_wait(&bars[1], ph_mma, abortf);
        ph_mma ^= 1;
        tc_fence_after();
        if (want_dx) {
            float* orow = reinterpret_cast<float*>(bufX) + (size_t)prow * K;
#pragma unroll 1
            for (int c8 = half; c8 < nchK; c8 += kHalves) {
                float u[8];
                tmem_ld8(tmem_addr(tDX, qtr, 8 * c8), u);
                tmem_wait_ld();
                if (valid) st8<VEC>(orow, 8 * c8, K, u);
            }
            tc_fence_before();
            fence_async_smem();
            __syncthreads();
            if (warp == 0) {
                if (lane == 0) bulk_s2g(a.out + (size_t)tile * 128 * K, bufX, (uint32_t)nrows * K * 4u);
                bulk_commit();
            }
        }
    }
    if (warp == 0) bulk_wait_all0();
    __syncthreads();
    if (!first) {
        float* stg = reinterpret_cast<float*>(bufX);          // [KP][KP+1]
        constexpr int SP = KP + 1;
        tc_fence_after();
#pragma unroll 1
        for (int c8 = half; c8 < NCH; c8 += kHalves) {
            float u[8];
            tmem_ld8(tmem_addr(tDW, qtr, 8 * c8), u);
            tmem_wait_ld();
            if (prow < KP)
#pragma unroll
                for (int j = 0; j < 8; ++j) stg[prow * SP + 8 * c8 + j] = u[j];
        }
        __syncthreads();
        for (int i = tid; i < N * K; i += kCtaThreads) {
            const int n = i / K, k = i - n * K;
            red_add(a.g_w + i, stg[n * SP + k]);
        }
        for (int n = tid; n < N; n += kCtaThreads) red_add(a.g_b + n, stg[n * SP + K]);
    }
    cta_end<TM_COLS>(abortf, a.abort_count, tmem, tid);
}

}  // namespace lin
}  // namespace mmx
