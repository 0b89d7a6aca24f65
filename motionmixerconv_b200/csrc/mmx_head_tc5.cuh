// MlpMixer output head on the Blackwell tensor cores (tcgen05 + TMEM + bulk-copy engine), sm_100a, ONE kernel per direction:
//
//     out = fc_out(conv_out(LN(x)))          x: [B,T,H] -> out: [B,To,D]
//     reference: h36m/mlp_mixer.py:332-335 (LayerNorm, Conv1d(seq_len, pred_len, 1) over the frames, Linear(H, D));
//     restated in oracle/mixer_np.py.
//
// A tile is S = 128 / max(T,To) whole sequences: S*T input rows, S*To output rows, one thread (TMEM lane) per row.  The mixing
// over the frames crosses rows, i.e. threads -- so it runs on the tensor core as a product with the BLOCK-DIAGONAL matrix
// Wbd[(s,o)][(s',t)] = [s == s'] conv_out.weight[o][t]  (128 x 128, staged once per CTA):
//     P = Wbd Z            Z = LN(x) rows, MN-major operand (K = rows)
//     out = P Wf^T + bf
// Backward (forward recomputed): dP = dOut Wf, dWf += dOut^T [P | 1], dZ = Wbd^T dP, and the time-mix weight gradient comes
// out of G += dP Z^T (128 x 128, accumulated in TMEM over the CTA's tiles) whose diagonal blocks are summed at the end.
// All products use bf16 hi+lo split operands (three MMAs each, fp32 accumulation): the bf16x3 toolkit of mmx_tc5.cuh.
#pragma once
#include "mmx_tc5.cuh"

namespace mmx {
namespace head {

using namespace tc5;

constexpr int KH = 64;     // padded hidden width: H + 1 <= KH (the ones column of the bias gradient)
constexpr int KD = 80;     // padded output width: D <= KD
using PH = Panels<KH>;      // operands with H-wide rows
using PD = Panels<KD>;      // operands with D-wide rows, and the weight Wf [D][H]
using PB = Panels<128>;     // block-diagonal time-mix matrix 128 x 128
constexpr uint32_t PS = PH::PS;
constexpr int CPT = KH / 8 / kHalves;                               // chunks of a hidden row per thread
static_assert(CPT * kHalves * 8 == KH, "KH must split evenly over the halves");

struct HeadArgs {
    const float* x;        // [B,T,H]
    const float* dout;     // backward: [B,To,D]
    float* out;            // forward: [B,To,D]; backward: dx [B,T,H]
    const float *ln_g, *ln_b, *wt, *bt, *wf, *bf;
    float *g_ln_g, *g_ln_b, *g_wt, *g_bt, *g_wf, *g_bf;
    int B, T, To, H, D, S;
    int* abort_count;
};

constexpr uint32_t kSmallFloats = 128 + KD + 2 * KH + 4 * kHalves * 128 + 2 * KH + 128 + 64;   // bt per row | bf | gamma, beta | exchange | dgamma, dbeta | dbt | barriers

struct HeadSmem {
    uint32_t x, y, o, wbd, wf, s1, small, total;
};
MMX_HD HeadSmem head_smem(int H, int D, bool bwd) {
    HeadSmem m;
    const uint32_t st_in = up128(128u * H * 4u + 64u), st_out = up128(128u * D * 4u + 64u);
    uint32_t o = 0;
    m.x = o; o += bwd ? umax(PH::BUF, st_in) : umax(PH::BUF, st_out);   // Z operand; doubles as the output staging tile
    m.y = o; o += bwd ? umax(PH::BUF, st_out) : PH::BUF;                // P operand (backward: also the landing zone of the dOut tile)
    m.o = o; o += bwd ? umax(PD::BUF, st_in) : 0;                       // backward: dOut / dP operand (also the landing zone of the x tile)
    m.wbd = o; o += PB::BUF;
    m.wf = o; o += PD::WBUF;
    m.s1 = o; o += bwd ? 0 : st_in;                                     // forward: x tile
    m.small = o; o += kSmallFloats * 4;
    m.total = o + 1024;
    return m;
}

struct Small {
    float *btrow, *bf, *gam, *bet, *ex, *dgam, *dbet, *dbt;
    uint64_t* bars;
    uint32_t* tslot;
    volatile int* abortf;
    MMX_D explicit Small(uint8_t* p) {
        btrow = reinterpret_cast<float*>(p);
        bf = btrow + 128;
        gam = bf + KD;
        bet = gam + KH;
        ex = bet + KH;
        dgam = ex + 4 * kHalves * 128;
        dbet = dgam + KH;
        dbt = dbet + KH;
        bars = reinterpret_cast<uint64_t*>(dbt + 128);
        tslot = reinterpret_cast<uint32_t*>(bars + 4);
        abortf = reinterpret_cast<volatile int*>(tslot + 1);
    }
};

// parameters -> shared memory.  Contains CTA barriers.
MMX_D void head_prologue(const HeadArgs& a, uint8_t* wbd, uint8_t* wfb, const Small& sm, int tid) {
    const int T = a.T, To = a.To, S = a.S;
    for (int i = tid; i < (int)((PB::BUF + PD::WBUF) / 16); i += kCtaThreads) reinterpret_cast<uint4*>(wbd)[i] = make_uint4(0, 0, 0, 0);   // wbd, wf contiguous
    for (int r = tid; r < 128; r += kCtaThreads) { sm.btrow[r] = r < S * To ? a.bt[r % To] : 0.0f; sm.dbt[r] = 0.0f; }
    for (int c = tid; c < KD; c += kCtaThreads) sm.bf[c] = c < a.D ? a.bf[c] : 0.0f;
    for (int c = tid; c < KH; c += kCtaThreads) {
        sm.gam[c] = c < a.H ? a.ln_g[c] : 0.0f;
        sm.bet[c] = c < a.H ? a.ln_b[c] : 0.0f;
        sm.dgam[c] = 0.0f;
        sm.dbet[c] = 0.0f;
    }
    __syncthreads();
    stage_weight<KD>(wfb, a.wf, a.D, a.H, nullptr, tid);
    for (int i = tid; i < S * To * T; i += kCtaThreads) {
        const int s = i / (To * T), ot = i - s * To * T, o = ot / T, t = ot - o * T;
        const int row = s * To + o, col = s * T + t;
        const Split sp = split1(a.wt[ot]);
        const uint32_t off = panel_off(row, col, PS);
        *reinterpret_cast<uint16_t*>(wbd + off) = (uint16_t)sp.hi;
        *reinterpret_cast<uint16_t*>(wbd + PB::PLANE + off) = (uint16_t)sp.lo;
    }
}

// LayerNorm statistics of the thread's row (shifted one-pass); the halves of a row exchange their partial sums
MMX_D void ln_row_stats(const float* srow, bool valid, int H, int half, int prow, float* ex, float& mean, float& rstd) {
    const int nchH = (H + 7) >> 3;
    const float c0 = valid ? srow[0] : 0.0f;
    float s = 0.0f, ss = 0.0f;
    if (valid) {
#pragma unroll 1
        for (int c8 = half; c8 < nchH; c8 += kHalves) {
            float v[8];
            ld8<2>(srow, 8 * c8, H, v);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float dv = 8 * c8 + j < H ? v[j] - c0 : 0.0f;
                s += dv;
                ss = fmaf(dv, dv, ss);
            }
        }
    }
    row_exchange(ex, half, prow, s, ss);
    const float ms = s / (float)H;
    mean = c0 + ms;
    rstd = 1.0f / sqrtf(fmaxf(ss / (float)H - ms * ms, 0.0f) + 1e-5f);
}

// ==========================================================================================
// forward
// ==========================================================================================
__global__ void __launch_bounds__(kCtaThreads) head_fwd_kernel(const HeadArgs a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const HeadSmem m = head_smem(a.H, a.D, false);
    uint8_t *bufX = base + m.x, *bufY = base + m.y, *wbd = base + m.wbd, *wfb = base + m.wf;
    float* S1 = reinterpret_cast<float*>(base + m.s1);
    const Small sm(base + m.small);
    uint64_t* bars = sm.bars;
    volatile int* abortf = sm.abortf;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, qtr = warp & 3, half = warp >> 2;
    const int prow = qtr * 32 + lane;
    const int T = a.T, To = a.To, H = a.H, D = a.D, S = a.S;
    constexpr int TM_COLS = 256;
    cta_begin<TM_COLS>(bars, 2, abortf, sm.tslot, tid);
    pdl_launch_dependents();
    head_prologue(a, wbd, wfb, sm, tid);
    pdl_wait();
    const int ntiles = (a.B + S - 1) / S;
    auto nseq_of = [&](int tile) { return min(S, a.B - tile * S); };
    auto load_x = [&](int tile) {
        const uint32_t bytes = (uint32_t)nseq_of(tile) * T * H * 4u;
        mbar_expect_tx(&bars[0], bytes);
        bulk_g2s(S1, a.x + (size_t)tile * S * T * H, bytes, &bars[0]);
    };
    if (tid == 0 && (int)blockIdx.x < ntiles) load_x(blockIdx.x);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *sm.tslot;
    const uint32_t tP = tmem, tO = tmem + KH;
    const uint32_t xB = smem_u32(bufX), yB = smem_u32(bufY), bdB = smem_u32(wbd), wfB = smem_u32(wfb);
    uint32_t ph_in = 0, ph_mma = 0;
    const int nchD = (D + 7) >> 3;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int nseq = nseq_of(tile);
        const bool vin = prow < nseq * T, vout = prow < nseq * To;
        const float* srow = S1 + (size_t)prow * H;
        mbar_wait(&bars[0], ph_in, abortf);
        ph_in ^= 1;
        if (warp == 0) bulk_wait_read0();              // the previous tile's output (staged in the X region) has left shared memory
        float mean, rstd;
        ln_row_stats(srow, vin, H, half, prow, sm.ex, mean, rstd);
        // ---------------- P0: Z = LN(x) -> operand X
#pragma unroll 1
        for (int c8 = half; c8 < KH / 8; c8 += kHalves) {
            float v[8], g[8], b[8];
            ld8<2>(srow, 8 * c8, vin ? H : 0, v);
            ld8s(sm.gam + 8 * c8, g);
            ld8s(sm.bet + 8 * c8, b);
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = (vin && 8 * c8 + j < H) ? fmaf((v[j] - mean) * rstd, g[j], b[j]) : 0.0f;
            put_chunk(bufX, PH::PLANE, PS, prow, c8, v);
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            const int next = tile + gridDim.x;
            if (next < ntiles) load_x(next);
            tc_fence_after();
            // P[(s,o)][h] = sum_(s',t) Wbd[(s,o)][(s',t)] Z[(s',t)][h]     (A K-major, B = Z read MN-major: K = rows)
            gemm3<0, 1>(tP, bdB, bdB + PB::PLANE, PS, xB, xB + PH::PLANE, PS, KH, 128 / 16, false);
            mma_commit(&bars[1]);
        }
        // ---------------- E1: P + bt -> operand Y
        mbar_wait(&bars[1], ph_mma, abortf);
        ph_mma ^= 1;
        tc_fence_after();
        {
            const float bt = sm.btrow[prow];
#pragma unroll 1
            for (int c8 = half; c8 < KH / 8; c8 += kHalves) {
                float u[8];
                tmem_ld8(tmem_addr(tP, qtr, 8 * c8), u);
                tmem_wait_ld();
#pragma unroll
                for (int j = 0; j < 8; ++j) u[j] = (vout && 8 * c8 + j < H) ? u[j] + bt : 0.0f;
                put_chunk(bufY, PH::PLANE, PS, prow, c8, u);
            }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            gemm3<0, 0>(tO, yB, yB + PH::PLANE, PS, wfB, wfB + PD::WPLANE, PD::WPS, KD, KH / 16, false);
            mma_commit(&bars[1]);
        }
        // ---------------- E2: out = . + bf -> staged rows -> global
        mbar_wait(&bars[1], ph_mma, abortf);
        ph_mma ^= 1;
        tc_fence_after();
        {
            float* orow = reinterpret_cast<float*>(bufX) + (size_t)prow * D;
#pragma unroll 1
            for (int c8 = half; c8 < nchD; c8 += kHalves) {
                float u[8], b[8];
                tmem_ld8(tmem_addr(tO, qtr, 8 * c8), u);
                ld8s(sm.bf + 8 * c8, b);
                tmem_wait_ld();
#pragma unroll
                for (int j = 0; j < 8; ++j) u[j] += b[j];
                if (vout) st8<2>(orow, 8 * c8, D, u);
            }
        }
        tc_fence_before();
        fence_async_smem();
        __syncthreads();
        if (tid == 0) {
            bulk_s2g(a.out + (size_t)tile * S * To * D, bufX, (uint32_t)nseq * To * D * 4u);
            bulk_commit();
        }
    }
    cta_end<TM_COLS>(abortf, a.abort_count, tmem, tid);
}

// ==========================================================================================
// backward
// ==========================================================================================
__global__ void __launch_bounds__(kCtaThreads) head_bwd_kernel(const HeadArgs a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const HeadSmem m = head_smem(a.H, a.D, true);
    uint8_t *bufX = base + m.x, *bufY = base + m.y, *bufO = base + m.o, *wbd = base + m.wbd, *wfb = base + m.wf;
    float* S1 = reinterpret_cast<float*>(bufO);       // x tile lands in the O region
    float* S2 = reinterpret_cast<float*>(bufY);       // dOut tile lands in the Y region
    const Small sm(base + m.small);
    uint64_t* bars = sm.bars;
    volatile int* abortf = sm.abortf;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, qtr = warp & 3, half = warp >> 2;
    const int prow = qtr * 32 + lane;
    const int T = a.T, To = a.To, H = a.H, D = a.D, S = a.S;
    constexpr int TM_COLS = 512;
    cta_begin<TM_COLS>(bars, 2, abortf, sm.tslot, tid);
    pdl_launch_dependents();
    head_prologue(a, wbd, wfb, sm, tid);
    pdl_wait();
    const int ntiles = (a.B + S - 1) / S;
    auto nseq_of = [&](int tile) { return min(S, a.B - tile * S); };
    auto load_tile = [&](int tile) {
        const uint32_t bx = (uint32_t)nseq_of(tile) * T * H * 4u, bd = (uint32_t)nseq_of(tile) * To * D * 4u;
        mbar_expect_tx(&bars[0], bx + bd);
        bulk_g2s(S1, a.x + (size_t)tile * S * T * H, bx, &bars[0]);
        bulk_g2s(S2, a.dout + (size_t)tile * S * To * D, bd, &bars[0]);
    };
    if (tid == 0 && (int)blockIdx.x < ntiles) load_tile(blockIdx.x);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *sm.tslot;
    // P / dZ | dP | xhat (parked) | dWf [d][h | ones] | G [(s,o)][(s',t)]
    const uint32_t tP = tmem, tDP = tmem + KH, tXH = tmem + 2 * KH, tDWF = tmem + 3 * KH, tG = tmem + 4 * KH;
    const uint32_t xB = smem_u32(bufX), yB = smem_u32(bufY), oB = smem_u32(bufO), bdB = smem_u32(wbd), wfB = smem_u32(wfb);
    uint32_t ph_in = 0, ph_mma = 0;
    bool first = true;
    float accG[CPT][8], accB[CPT][8];           // dLN.weight / dLN.bias partial sums of the thread's columns over its rows
#pragma unroll
    for (int i = 0; i < CPT; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) accG[i][j] = accB[i][j] = 0.0f;
    float dbt_acc = 0.0f;

    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int nseq = nseq_of(tile);
        const bool vin = prow < nseq * T, vout = prow < nseq * To;
        const float* srow = S1 + (size_t)prow * H;
        const float* drow = S2 + (size_t)prow * D;
        mbar_wait(&bars[0], ph_in, abortf);
        ph_in ^= 1;
        if (warp == 0) bulk_wait_read0();              // the previous tile's dx (staged in the X region) has left shared memory
        float mean, rstd;
        ln_row_stats(srow, vin, H, half, prow, sm.ex, mean, rstd);
        // ---------------- P0: Z = LN(x) -> operand X; xhat -> TMEM
#pragma unroll 1
        for (int c8 = half; c8 < KH / 8; c8 += kHalves) {
            float v[8], z[8], g[8], b[8];
            ld8<2>(srow, 8 * c8, vin ? H : 0, v);
            ld8s(sm.gam + 8 * c8, g);
            ld8s(sm.bet + 8 * c8, b);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const bool ok = vin && 8 * c8 + j < H;
                v[j] = ok ? (v[j] - mean) * rstd : 0.0f;
                z[j] = ok ? fmaf(v[j], g[j], b[j]) : 0.0f;
            }
            put_chunk(bufX, PH::PLANE, PS, prow, c8, z);
            tmem_st8(tmem_addr(tXH, qtr, 8 * c8), v);
        }
        tmem_wait_st();
        fence_async_smem();
        tc_fence_before();
        __syncthreads();           // operand X complete; the x tile (O region) is consumed
        if (tid == 0) {
            tc_fence_after();
            gemm3<0, 1>(tP, bdB, bdB + PB::PLANE, PS, xB, xB + PH::PLANE, PS, KH, 128 / 16, false);
            mma_commit(&bars[1]);
        }
        // ---------------- P1: dOut -> operand O
#pragma unroll 1
        for (int c8 = half; c8 < KD / 8; c8 += kHalves) {
            float v[8];
            ld8<2>(drow, 8 * c8, vout ? D : 0, v);
            put_chunk(bufO, PD::PLANE, PS, prow, c8, v);
        }
        __syncthreads();           // the dOut tile (Y region) is consumed
        // ---------------- E1: P + bt (+ ones column at H) -> operand Y
        mbar_wait(&bars[1], ph_mma, abortf);
        ph_mma ^= 1;
        tc_fence_after();
        {
            const float bt = sm.btrow[prow];
#pragma unroll 1
            for (int c8 = half; c8 < KH / 8; c8 += kHalves) {
                float u[8];
                tmem_ld8(tmem_addr(tP, qtr, 8 * c8), u);
                tmem_wait_ld();
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int c = 8 * c8 + j;
                    u[j] = !vout ? 0.0f : (c < H ? u[j] + bt : (c == H ? 1.0f : 0.0f));
                }
                put_chunk(bufY, PH::PLANE, PS, prow, c8, u);
            }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            // dP = dOut Wf                 (A = dOut K-major, B = Wf [D rows][H cols] read MN-major: K = d)
            gemm3<0, 1>(tDP, oB, oB + PD::PLANE, PS, wfB, wfB + PD::WPLANE, PD::WPS, KH, KD / 16, false);
            // dWf[d][h] += sum_r dOut[r][d] P[r][h]   (both MN-major, K = the 128 rows); column H of P is all ones -> dbf
            gemm3<1, 1>(tDWF, oB, oB + PD::PLANE, PS, yB, yB + PH::PLANE, PS, KH, 128 / 16, !first);
            mma_commit(&bars[1]);
        }
        // ---------------- E2: dP -> operand O (over dOut); its row sums -> dbt
        mbar_wait(&bars[1], ph_mma, abortf);
        ph_mma ^= 1;
        tc_fence_after();
#pragma unroll 1
        for (int c8 = half; c8 < KH / 8; c8 += kHalves) {
            float u[8];
            tmem_ld8(tmem_addr(tDP, qtr, 8 * c8), u);
            tmem_wait_ld();
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                u[j] = (vout && 8 * c8 + j < H) ? u[j] : 0.0f;
                dbt_acc += u[j];
            }
            put_chunk(bufO, PD::PLANE, PS, prow, c8, u);
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            // dZ[(s',t)][h] = sum_(s,o) Wbd[(s,o)][(s',t)] dP[(s,o)][h]     (A = Wbd read MN-major, B = dP read MN-major)
            gemm3<1, 1>(tP, bdB, bdB + PB::PLANE, PS, oB, oB + PD::PLANE, PS, KH, 128 / 16, false);
            // G[(s,o)][(s',t)] += sum_h dP[(s,o)][h] Z[(s',t)][h]           (both K-major)
            gemm3<0, 0>(tG, oB, oB + PD::PLANE, PS, xB, xB + PH::PLANE, PS, 128, KH / 16, !first);
            mma_commit(&bars[1]);
        }
        first = false;
        // ---------------- E3: LayerNorm backward -> staged dx rows
        mbar_wait(&bars[1], ph_mma, abortf);
        ph_mma ^= 1;
        tc_fence_after();
        if (tid == 0) {                                // the Y and O regions are free: fetch the next tile
            const int next = tile + gridDim.x;
            if (next < ntiles) load_tile(next);
        }
        {
            float dxh[CPT][8], xh[CPT][8];
            float m1 = 0.0f, m2 = 0.0f;
#pragma unroll
            for (int i = 0; i < CPT; ++i) {
                const int c8 = half + kHalves * i;
                float dz[8], g[8];
                tmem_ld8(tmem_addr(tP, qtr, 8 * c8), dz);
                tmem_ld8(tmem_addr(tXH, qtr, 8 * c8), xh[i]);
                ld8s(sm.gam + 8 * c8, g);
                tmem_wait_ld();
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float d = vin ? dz[j] : 0.0f;
                    accG[i][j] = fmaf(d, xh[i][j], accG[i][j]);
                    accB[i][j] += d;
                    dxh[i][j] = d * g[j];
                    m1 += dxh[i][j];
                    m2 = fmaf(dxh[i][j], xh[i][j], m2);
                }
            }
            row_exchange(sm.ex, half, prow, m1, m2);
            m1 /= (float)H;
            m2 /= (float)H;
            float* orow = reinterpret_cast<float*>(bufX) + (size_t)prow * H;
#pragma unroll
            for (int i = 0; i < CPT; ++i) {
                const int c8 = half + kHalves * i;
#pragma unroll
                for (int j = 0; j < 8; ++j) dxh[i][j] = rstd * (dxh[i][j] - m1 - xh[i][j] * m2);
                if (vin) st8<2>(orow, 8 * c8, H, dxh[i]);
            }
        }
        tc_fence_before();
        fence_async_smem();
        __syncthreads();
        if (tid == 0) {
            bulk_s2g(a.out + (size_t)tile * S * T * H, bufX, (uint32_t)nseq * T * H * 4u);
            bulk_commit();
        }
    }
    if (warp == 0) bulk_wait_all0();
    __syncthreads();

    // ---------------- flush
    if (!first) {
        tc_fence_after();
        // dLN.weight / dLN.bias: sum over the 32 rows of the warp, then one shared atomic per warp and column
#pragma unroll
        for (int i = 0; i < CPT; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float g = accG[i][j], b = accB[i][j];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) { g += __shfl_xor_sync(0xffffffffu, g, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
                const int c = 8 * (half + kHalves * i) + j;
                if (lane == 0 && c < H) { atomicAdd(sm.dgam + c, g); atomicAdd(sm.dbet + c, b); }
            }
        if (prow < S * To) atomicAdd(sm.dbt + prow % To, dbt_acc);
        // dWf, dbf: TMEM (lane = d) -> staging -> global
        float* stg = reinterpret_cast<float*>(bufX);          // [KD][KH+1]
        constexpr int SP = KH + 1;
#pragma unroll 1
        for (int c8 = half; c8 < KH / 8; c8 += kHalves) {
            float u[8];
            tmem_ld8(tmem_addr(tDWF, qtr, 8 * c8), u);
            tmem_wait_ld();
            if (prow < KD)
#pragma unroll
                for (int j = 0; j < 8; ++j) stg[prow * SP + 8 * c8 + j] = u[j];
        }
        // G: TMEM (lane = (s,o)) -> staging [128][128] with the columns rotated by the row (conflict-free stores)
        float* gst = reinterpret_cast<float*>(wbd);           // the time-mix operand is dead: 64 KB
#pragma unroll 1
        for (int c8 = half; c8 < 16; c8 += kHalves) {
            float u[8];
            tmem_ld8(tmem_addr(tG, qtr, 8 * c8), u);
            tmem_wait_ld();
#pragma unroll
            for (int j = 0; j < 8; ++j) gst[prow * 128 + ((8 * c8 + j + prow) & 127)] = u[j];
        }
        __syncthreads();
        for (int i = tid; i < D * H; i += kCtaThreads) {
            const int d = i / H, h = i - d * H;
            red_add(a.g_wf + i, stg[d * SP + h]);
        }
        for (int d = tid; d < D; d += kCtaThreads) red_add(a.g_bf + d, stg[d * SP + H]);
        for (int i = tid; i < To * T; i += kCtaThreads) {
            const int o = i / T, t = i - o * T;
            float v = 0.0f;
            for (int s = 0; s < S; ++s) {
                const int r = s * To + o;
                v += gst[r * 128 + ((s * T + t + r) & 127)];
            }
            red_add(a.g_wt + i, v);
        }
        for (int o = tid; o < To; o += kCtaThreads) red_add(a.g_bt + o, sm.dbt[o]);
        for (int h = tid; h < H; h += kCtaThreads) { red_add(a.g_ln_g + h, sm.dgam[h]); red_add(a.g_ln_b + h, sm.dbet[h]); }
    }
    cta_end<TM_COLS>(abortf, a.abort_count, tmem, tid);
}

}  // namespace head
}  // namespace mmx
