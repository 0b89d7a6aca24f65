// Channel half of a MixerBlock on the Blackwell tensor cores (tcgen05 + TMEM + bulk-copy engine), sm_100a.
//
//     y = x1 + SE(reg2(fc2(reg1(act(fc1(LN2(x1)))))))          reference: h36m/mlp_mixer.py:157-164 (MixerBlock.forward, second
//     half), MlpBlock :87-96, SELayer :30-34; restated in oracle/mixer_np.py (MlpMixerOracle.forward / backward).
//
// Work unit: a tile of 4 * (32 / T) whole sequences = one 128-row MMA tile.  Row r of the tile is TMEM lane r; the kHalves warps
// that may touch a lane quarter (warp % 4) split the row's 8-column chunks between them, so LayerNorm, the activation,
// dropout, the squeeze sum and the LayerNorm backward are per-thread loops over part of a row plus one shared-memory exchange
// of the partial sums.  The T frames of a sequence sit in T consecutive lanes of one warp: the SE excitation is a handful of
// shuffles.  Lanes 32/T*T .. 31 of every warp are padding rows (all-zero operands).
//
// Contractions and operands: the bf16x3 products on the 16-bit panel layout of mmx_tc5.cuh (read its header first).
// LN2's affine is folded into fc1 (W1' = W1 * gamma2, b1' = b1 + W1 beta2): the A operand is the plain normalised row and
// dgamma2, dbeta2, dW1 are derived at flush time from ONE accumulated product  Wt = dU^T xhat.  Bias gradients ride along as a
// column of ones in the B operand of the weight-gradient products.  dW1 / dW2 accumulate in TMEM across the CTA's whole
// persistent loop and are flushed once (no shared-memory accumulators, no locks).  Rows a thread needs again later in the
// tile (the residual input, xhat) are parked in spare TMEM columns, so every per-row loop is a rolled loop over chunks
// (small code: the first version, fully unrolled over register-resident rows, was 300 KB of SASS and instruction-fetch bound).
// Activations enter and leave through the bulk-copy engine (cp.async.bulk, SASS UBLKCP) with mbarrier completion.
#pragma once
#include "mmx_tc5.cuh"

namespace mmx {
namespace chan {

using namespace tc5;

constexpr int kMaxRR = 4;                      // SE bottleneck width served (T // r_se)

struct ChanArgs {
    const float* x1;               // [B*T, H]   input of the channel half
    const float* dy;               // [B*T, H]   upstream gradient (backward)
    float* out;                    // forward: y; backward: dx1
    const float *ln_g, *ln_b, *w1, *b1, *w2, *b2, *se1, *se2;
    float *g_ln_g, *g_ln_b, *g_w1, *g_b1, *g_w2, *g_b2, *g_se1, *g_se2;
    int B, T, H, ch, rr;           // rr = SE hidden width (0: no SE)
    int site_base;                 // dropout site of the block's first Dropout; the channel MLP uses site_base + 2 / + 3
    Dropout dr;
    int* abort_count;              // device counter, incremented if a pipeline wait times out (tests assert it stays 0)
};

struct Geo {
    int spw, rpw, seq_per_tile, tile_rows, pitch;
};
MMX_HD Geo make_geo(int T, int H, int vec) {
    Geo g;
    g.spw = 32 / T;
    g.rpw = g.spw * T;
    g.seq_per_tile = 4 * g.spw;
    g.tile_rows = 4 * g.rpw;
    g.pitch = vec == 4 ? H + 4 : H;
    return g;
}
// fp32 staging tile of one 128-row tile (+ slack: chunk loads of the last row may run past the row)
MMX_HD uint32_t stage_bytes(const Geo& g) { return up128((uint32_t)g.tile_rows * g.pitch * 4u + 64u); }

// shared-memory layout (byte offsets from the 1024-aligned base; total includes the alignment slack)
struct ChanSmem {
    uint32_t x, y, w1, w2, s1, s2, small, total;
};
template <int KP>
MMX_HD ChanSmem chan_smem(const Geo& g, bool bwd) {
    using P = Panels<KP>;
    const uint32_t st = stage_bytes(g), buf = umax(P::BUF, st);    // the X region doubles as the output staging tile
    ChanSmem m;
    uint32_t o = 0;
    m.x = o; o += buf;
    m.y = bwd ? o : m.x; o += bwd ? buf : 0;                        // backward: second operand
    m.w1 = o; o += P::WBUF;
    m.w2 = o; o += P::WBUF;
    m.s1 = o; o += st;                                              // x1 tile
    m.s2 = bwd ? o : m.s1; o += bwd ? st : 0;                       // backward: dy tile
    m.small = o; o += (4 * KP + 2 * 32 * kMaxRR + 4 * kHalves * 128 + 64) * 4;   // c1f, c2, gamma2, spare | se1, se2 | exchange | barriers
    m.total = o + 1024;
    return m;
}

// per-CTA constants: weights (LN2 affine folded into fc1), biases, SE weights.  Contains CTA barriers.
template <int KP>
MMX_D void prologue(const ChanArgs& a, uint8_t* w1b, uint8_t* w2b, float* c1f, float* c2, float* gam, float* se1, float* se2, int tid) {
    const int H = a.H, ch = a.ch, T = a.T, rr = a.rr;
    for (int i = tid; i < (int)(2 * Panels<KP>::WBUF / 16); i += kCtaThreads) reinterpret_cast<uint4*>(w1b)[i] = make_uint4(0, 0, 0, 0);   // w1b, w2b contiguous
    for (int c = tid; c < KP; c += kCtaThreads) {
        c2[c] = c < H ? a.b2[c] : 0.0f;
        gam[c] = c < H ? a.ln_g[c] : 0.0f;
        c1f[c] = 0.0f;
    }
    for (int i = tid; i < 32 * kMaxRR; i += kCtaThreads) {
        se1[i] = (rr > 0 && i < rr * T) ? a.se1[i] : 0.0f;
        se2[i] = (rr > 0 && i < rr * T) ? a.se2[i] : 0.0f;
    }
    __syncthreads();
    stage_weight<KP>(w1b, a.w1, ch, H, a.ln_g, tid);
    stage_weight<KP>(w2b, a.w2, H, ch, nullptr, tid);
    // b1'[c] = b1[c] + sum_h W1[c][h] beta2[h]: one warp per row, lanes over h
    const int warp = tid >> 5, lane = tid & 31;
    for (int c = warp; c < ch; c += kCtaThreads / 32) {
        float s = 0.0f;
        for (int h = lane; h < H; h += 32) s = fmaf(a.w1[(size_t)c * H + h], a.ln_b[h], s);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) c1f[c] = s + a.b1[c];
    }
}

// SE excitation of the sequence this lane belongs to (lanes seq_base .. seq_base+T-1 hold the T squeeze values)
struct SeOut { float gate; float z[kMaxRR]; };
MMX_D SeOut se_excite(float s, int t, int seq_base, int T, int rr, const float* se1, const float* se2) {
    SeOut o;
#pragma unroll
    for (int k = 0; k < kMaxRR; ++k) o.z[k] = 0.0f;
    for (int tt = 0; tt < T; ++tt) {
        const float v = __shfl_sync(0xffffffffu, s, seq_base + tt);
#pragma unroll
        for (int k = 0; k < kMaxRR; ++k)
            if (k < rr) o.z[k] = fmaf(se1[k * T + tt], v, o.z[k]);
    }
    float q = 0.0f;
#pragma unroll
    for (int k = 0; k < kMaxRR; ++k)
        if (k < rr) q = fmaf(se2[t * rr + k], fmaxf(o.z[k], 0.0f), q);
    o.gate = sigmoidf_(q);
    return o;
}

// pointers into the dynamic shared memory
template <int KP>
struct Carve {
    uint8_t *bufX, *bufY, *w1b, *w2b;
    float *S1, *S2, *c1f, *c2, *gam, *se1, *se2, *ex;
    uint64_t* bars;
    uint32_t* tslot;
    volatile int* abortf;
    MMX_D Carve(uint8_t* raw, const Geo& g, bool bwd) {
        uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~(uintptr_t)1023);
        const ChanSmem m = chan_smem<KP>(g, bwd);
        bufX = sm + m.x;
        bufY = sm + m.y;
        w1b = sm + m.w1;
        w2b = sm + m.w2;
        S1 = reinterpret_cast<float*>(sm + m.s1);
        S2 = reinterpret_cast<float*>(sm + m.s2);
        c1f = reinterpret_cast<float*>(sm + m.small);
        c2 = c1f + KP;
        gam = c2 + KP;
        se1 = gam + 2 * KP;
        se2 = se1 + 32 * kMaxRR;
        ex = se2 + 32 * kMaxRR;
        bars = reinterpret_cast<uint64_t*>(ex + 4 * kHalves * 128);
        tslot = reinterpret_cast<uint32_t*>(bars + 4);
        abortf = reinterpret_cast<volatile int*>(tslot + 1);
    }
};

// ==========================================================================================
// forward
// ==========================================================================================
template <int ACT, int KP, int VEC>
__global__ void __launch_bounds__(kCtaThreads) chan_fwd_kernel(const ChanArgs a) {
    using P = Panels<KP>;
    extern __shared__ uint8_t smem_raw[];
    const Geo g = make_geo(a.T, a.H, VEC);
    Carve<KP> cv(smem_raw, g, false);
    uint8_t* bufX = cv.bufX;
    float* S = cv.S1;
    uint64_t* bars = cv.bars;
    volatile int* abortf = cv.abortf;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, qtr = warp & 3, half = warp >> 2;
    const int prow = qtr * 32 + lane;
    const int H = a.H, ch = a.ch, T = a.T, rr = a.rr;
    const Dropout dr = resolve_dropout(a.dr);
    const uint32_t th16 = dr.thresh >> 16;
    const uint32_t key2 = drop_key(dr.seed_lo, dr.seed_hi, a.site_base + 2, dr.step), key3 = drop_key(dr.seed_lo, dr.seed_hi, a.site_base + 3, dr.step);
    constexpr int TM_COLS = 3 * KP <= 256 ? 256 : 512;
    constexpr int NCH = KP / 8;

    cta_begin<TM_COLS>(bars, 2, abortf, cv.tslot, tid);   // bars: X1 tile landed | MMA group done
    pdl_launch_dependents();
    const int ntiles = (a.B + g.seq_per_tile - 1) / g.seq_per_tile;
    auto tile_nrows = [&](int tile) { return min(g.seq_per_tile, a.B - tile * g.seq_per_tile) * a.T; };
    prologue<KP>(a, cv.w1b, cv.w2b, cv.c1f, cv.c2, cv.gam, cv.se1, cv.se2, tid);   // parameters only: overlaps the previous kernel's tail
    pdl_wait();                // the previous kernel (the token half) has completed: x1 is readable
    if (warp == 0 && (int)blockIdx.x < ntiles)
        stage_in<VEC>(S, a.x1, (size_t)blockIdx.x * g.tile_rows, tile_nrows(blockIdx.x), a.H, g.pitch, &bars[0], lane);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *cv.tslot;
    const uint32_t tU = tmem, tY = tmem + KP, tXR = tmem + 2 * KP;
    const uint32_t xB = smem_u32(bufX), w1B = smem_u32(cv.w1b), w2B = smem_u32(cv.w2b);

    const bool lane_ok = lane < g.rpw;
    const int t = lane_ok ? lane % T : 0;
    const int seq_base = lane_ok ? (lane / T) * T : 0;
    const int drow = qtr * g.rpw + (lane_ok ? lane : 0);
    const int nchH = (H + 7) >> 3;
    const uint32_t ch8 = (uint32_t)(ch + 7) >> 3, H8 = (uint32_t)nchH;
    uint32_t ph_in = 0, ph_mma = 0;

    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int nrows = tile_nrows(tile);
        const bool valid = lane_ok && drow < nrows;
        const uint32_t grow = (uint32_t)((size_t)tile * g.tile_rows + drow);
        const float* srow = S + (size_t)drow * g.pitch;

        // ---------------- P0: LayerNorm statistics (shifted one-pass), xhat -> operand X, raw row -> TMEM
        mbar_wait(&bars[0], ph_in, abortf);
        ph_in ^= 1;
        float mean, rstd;
        {
            const float c0 = valid ? srow[0] : 0.0f;
            float s = 0.0f, ss = 0.0f;
            if (valid) {
#pragma unroll 1
                for (int c8 = half; c8 < nchH; c8 += kHalves) {
                    float v[8];
                    ld8<VEC>(srow, 8 * c8, H, v);
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float dv = 8 * c8 + j < H ? v[j] - c0 : 0.0f;
                        s += dv;
                        ss = fmaf(dv, dv, ss);
                    }
                }
            }
            if (warp == 0) bulk_wait_read0();          // the previous tile's output (staged in the X region) has left shared memory
            row_exchange(cv.ex, half, prow, s, ss);
            const float ms = s / (float)H;
            mean = c0 + ms;
            rstd = 1.0f / sqrtf(fmaxf(ss / (float)H - ms * ms, 0.0f) + 1e-5f);
        }
#pragma unroll 1
        for (int c8 = half; c8 < NCH; c8 += kHalves) {
            float v[8], xh[8];
            ld8<VEC>(srow, 8 * c8, valid ? H : 0, v);
#pragma unroll
            for (int j = 0; j < 8; ++j) xh[j] = (valid && 8 * c8 + j < H) ? (v[j] - mean) * rstd : 0.0f;
            put_chunk(bufX, P::PLANE, P::PS, prow, c8, xh);
            tmem_st8(tmem_addr(tXR, qtr, 8 * c8), v);
        }
        tmem_wait_st();
        fence_async_smem();
        tc_fence_before();
        __syncthreads();       // operand X complete; S fully consumed
        if (warp == 0) {
            const int next = tile + gridDim.x;
            if (next < ntiles) stage_in<VEC>(S, a.x1, (size_t)next * g.tile_rows, tile_nrows(next), H, g.pitch, &bars[0], lane);
        }
        if (tid == 0) {
            tc_fence_after();
            gemm3<0, 0>(tU, xB, xB + P::PLANE, P::PS, w1B, w1B + P::WPLANE, P::WPS, KP, KP / 16, false);
            mma_commit(&bars[1]);
        }
        // ---------------- E1: U -> G = reg1(act(U + b1')) -> operand X
        mbar_wait(&bars[1], ph_mma, abortf);
        ph_mma ^= 1;
        tc_fence_after();
#pragma unroll 1
        for (int c8 = half; c8 < NCH; c8 += kHalves) {
            float u[8], b[8];
            tmem_ld8(tmem_addr(tU, qtr, 8 * c8), u);
            ld8s(cv.c1f + 8 * c8, b);
            const uint32_t kb = th16 ? keep8(key2, th16, grow, ch8, c8) : 0xffu;
            tmem_wait_ld();
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float gv = act_fwd<ACT>(u[j] + b[j]);
                gv = (kb >> j) & 1u ? gv * dr.scale : 0.0f;
                u[j] = (valid && 8 * c8 + j < ch) ? gv : 0.0f;
            }
            put_chunk(bufX, P::PLANE, P::PS, prow, c8, u);
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            gemm3<0, 0>(tY, xB, xB + P::PLANE, P::PS, w2B, w2B + P::WPLANE, P::WPS, KP, KP / 16, false);
            mma_commit(&bars[1]);
        }
        // ---------------- E2: Y2 -> reg2 -> SE -> + residual -> staged output row
        mbar_wait(&bars[1], ph_mma, abortf);
        ph_mma ^= 1;
        tc_fence_after();
        float ssum = 0.0f, dummy = 0.0f;
#pragma unroll 1
        for (int c8 = half; c8 < nchH; c8 += kHalves) {
            float u[8], b[8];
            tmem_ld8(tmem_addr(tY, qtr, 8 * c8), u);
            ld8s(cv.c2 + 8 * c8, b);
            const uint32_t kb = th16 ? keep8(key3, th16, grow, H8, c8) : 0xffu;
            tmem_wait_ld();
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float yv = u[j] + b[j];
                yv = (kb >> j) & 1u ? yv * dr.scale : 0.0f;
                yv = (valid && 8 * c8 + j < H) ? yv : 0.0f;
                u[j] = yv;
                ssum += yv;
            }
            tmem_st8(tmem_addr(tY, qtr, 8 * c8), u);
        }
        tmem_wait_st();
        row_exchange(cv.ex, half, prow, ssum, dummy);
        float gate = 1.0f;
        if (rr > 0) gate = se_excite(ssum / (float)H, t, seq_base, T, rr, cv.se1, cv.se2).gate;
        {
            float* orow = reinterpret_cast<float*>(bufX) + (size_t)drow * g.pitch;
#pragma unroll 1
            for (int c8 = half; c8 < nchH; c8 += kHalves) {
                float y[8], x[8];
                tmem_ld8(tmem_addr(tY, qtr, 8 * c8), y);
                tmem_ld8(tmem_addr(tXR, qtr, 8 * c8), x);
                tmem_wait_ld();
#pragma unroll
                for (int j = 0; j < 8; ++j) y[j] = fmaf(y[j], gate, x[j]);
                if (valid) st8<VEC>(orow, 8 * c8, H, y);
            }
        }
        tc_fence_before();
        fence_async_smem();
        __syncthreads();
        if (warp == 0) stage_out<VEC>(a.out, reinterpret_cast<const float*>(bufX), (size_t)tile * g.tile_rows, nrows, H, g.pitch, lane);
    }
    cta_end<TM_COLS>(abortf, a.abort_count, tmem, tid);
}

// ==========================================================================================
// backward (forward recomputed from x1)
// ==========================================================================================
template <int ACT, int KP, int VEC>
__global__ void __launch_bounds__(kCtaThreads) chan_bwd_kernel(const ChanArgs a) {
    using P = Panels<KP>;
    extern __shared__ uint8_t smem_raw[];
    const Geo g = make_geo(a.T, a.H, VEC);
    Carve<KP> cv(smem_raw, g, true);
    uint8_t* bufX = cv.bufX;                  // xhat -> dY2 -> xhat again -> output staging
    uint8_t* bufY = cv.bufY;                  // G2 -> dU2
    float* S1 = cv.S1;                        // x1 tile
    float* S2 = cv.S2;                        // dy tile
    uint64_t* bars = cv.bars;
    volatile int* abortf = cv.abortf;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, qtr = warp & 3, half = warp >> 2;
    const int prow = qtr * 32 + lane;
    const int H = a.H, ch = a.ch, T = a.T, rr = a.rr;
    const Dropout dr = resolve_dropout(a.dr);
    const uint32_t th16 = dr.thresh >> 16;
    const uint32_t key2 = drop_key(dr.seed_lo, dr.seed_hi, a.site_base + 2, dr.step), key3 = drop_key(dr.seed_lo, dr.seed_hi, a.site_base + 3, dr.step);
    constexpr int TM_COLS = 512;
    static_assert(5 * KP <= 512, "TMEM: five KP-column regions");
    constexpr int NCH = KP / 8;

    cta_begin<TM_COLS>(bars, 3, abortf, cv.tslot, tid);   // bars: x1 tile landed | MMA group done | dy tile landed
    pdl_launch_dependents();
    const int ntiles = (a.B + g.seq_per_tile - 1) / g.seq_per_tile;
    auto tile_nrows = [&](int tile) { return min(g.seq_per_tile, a.B - tile * g.seq_per_tile) * a.T; };
    prologue<KP>(a, cv.w1b, cv.w2b, cv.c1f, cv.c2, cv.gam, cv.se1, cv.se2, tid);   // parameters only: overlaps the previous kernel's tail
    pdl_wait();                // the previous kernel has completed: x1 / dy are readable, the gradient buffers may be added to
    if (warp == 0 && (int)blockIdx.x < ntiles) {
        stage_in<VEC>(S1, a.x1, (size_t)blockIdx.x * g.tile_rows, tile_nrows(blockIdx.x), a.H, g.pitch, &bars[0], lane);
        stage_in<VEC>(S2, a.dy, (size_t)blockIdx.x * g.tile_rows, tile_nrows(blockIdx.x), a.H, g.pitch, &bars[2], lane);
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *cv.tslot;
    // U2 / d xhat | Y2 / dG2 | xhat (parked) | Wt = dU^T xhat | dW2
    const uint32_t tU = tmem, tY = tmem + KP, tXH = tmem + 2 * KP, tDW1 = tmem + 3 * KP, tDW2 = tmem + 4 * KP;
    const uint32_t xB = smem_u32(bufX), yB = smem_u32(bufY), w1B = smem_u32(cv.w1b), w2B = smem_u32(cv.w2b);

    const bool lane_ok = lane < g.rpw;
    const int t = lane_ok ? lane % T : 0;
    const int seq_base = lane_ok ? (lane / T) * T : 0;
    const int drow = qtr * g.rpw + (lane_ok ? lane : 0);
    const int nchH = (H + 7) >> 3;
    const uint32_t ch8 = (uint32_t)(ch + 7) >> 3, H8 = (uint32_t)nchH;
    uint32_t ph_x = 0, ph_dy = 0, ph_mma = 0;
    bool first = true;
    float gS1[kMaxRR], gS2[kMaxRR];
#pragma unroll
    for (int k = 0; k < kMaxRR; ++k) gS1[k] = gS2[k] = 0.0f;


    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int nrows = tile_nrows(tile);
        const bool valid = lane_ok && drow < nrows;
        const uint32_t grow = (uint32_t)((size_t)tile * g.tile_rows + drow);
        const int next = tile + gridDim.x;
        const float* srow = S1 + (size_t)drow * g.pitch;
        const float* drw = S2 + (size_t)drow * g.pitch;

        // ---------------- P0: xhat = LN2(x1) without affine (+ ones column at H) -> operand X and TMEM
        mbar_wait(&bars[0], ph_x, abortf);
        ph_x ^= 1;
        float mean, rstd;
        {
            const float c0 = valid ? srow[0] : 0.0f;
            float s = 0.0f, ss = 0.0f;
            if (valid) {
#pragma unroll 1
                for (int c8 = half; c8 < nchH; c8 += kHalves) {
                    float v[8];
                    ld8<VEC>(srow, 8 * c8, H, v);
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float dv = 8 * c8 + j < H ? v[j] - c0 : 0.0f;
                        s += dv;
                        ss = fmaf(dv, dv, ss);
                    }
                }
            }
            if (warp == 0) bulk_wait_read0();
            row_exchange(cv.ex, half, prow, s, ss);
            const float ms = s / (float)H;
            mean = c0 + ms;
            rstd = 1.0f / sqrtf(fmaxf(ss / (float)H - ms * ms, 0.0f) + 1e-5f);
        }
#pragma unroll 1
        for (int c8 = half; c8 < NCH; c8 += kHalves) {
            float v[8];
            ld8<VEC>(srow, 8 * c8, valid ? H : 0, v);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int k = 8 * c8 + j;
                v[j] = !valid ? 0.0f : (k < H ? (v[j] - mean) * rstd : (k == H ? 1.0f : 0.0f));
            }
            put_chunk(bufX, P::PLANE, P::PS, prow, c8, v);
            tmem_st8(tmem_addr(tXH, qtr, 8 * c8), v);
        }
        tmem_wait_st();
        fence_async_smem();
        tc_fence_before();
        __syncthreads();   // S1 consumed
        if (warp == 0 && next < ntiles) stage_in<VEC>(S1, a.x1, (size_t)next * g.tile_rows, tile_nrows(next), H, g.pitch, &bars[0], lane);
        if (tid == 0) {
            tc_fence_after();
            gemm3<0, 0>(tU, xB, xB + P::PLANE, P::PS, w1B, w1B + P::WPLANE, P::WPS, KP, KP / 16, false);
            mma_commit(&bars[1]);
        }
        // ---------------- E1: G2 = reg1(act(U2 + b1')) -> operand Y (ones column at ch); TMEM keeps reg1'(.) * act'(U2 + b1')
        // in place of U2 (what the backward needs of it), so the activation is evaluated once per element and tile
        mbar_wait(&bars[1], ph_mma, abortf);
        ph_mma ^= 1;
        tc_fence_after();
#pragma unroll 1
        for (int c8 = half; c8 < NCH; c8 += kHalves) {
            float u[8], b[8], dact[8];
            tmem_ld8(tmem_addr(tU, qtr, 8 * c8), u);
            ld8s(cv.c1f + 8 * c8, b);
            const uint32_t kb = th16 ? keep8(key2, th16, grow, ch8, c8) : 0xffu;
            tmem_wait_ld();
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int c = 8 * c8 + j;
                float gv;
                const float da = act_fwd_grad<ACT>(u[j] + b[j], &gv);
                const float ks = (kb >> j) & 1u ? dr.scale : 0.0f;
                dact[j] = (valid && c < ch) ? da * ks : 0.0f;
                u[j] = !valid ? 0.0f : (c < ch ? gv * ks : (c == ch ? 1.0f : 0.0f));
            }
            put_chunk(bufY, P::PLANE, P::PS, prow, c8, u);
            tmem_st8(tmem_addr(tU, qtr, 8 * c8), dact);
        }
        tmem_wait_st();
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            gemm3<0, 0>(tY, yB, yB + P::PLANE, P::PS, w2B, w2B + P::WPLANE, P::WPS, KP, KP / 16, false);
            mma_commit(&bars[1]);
        }
        // ---------------- E2: y2, SE forward + backward, dY2 -> operand X
        mbar_wait(&bars[2], ph_dy, abortf);
        ph_dy ^= 1;
        mbar_wait(&bars[1], ph_mma, abortf);
        ph_mma ^= 1;
        tc_fence_after();
        {
            float ssum = 0.0f, dgate = 0.0f;
            unsigned long long keepbits = 0ull;
            int i = 0;
#pragma unroll 1
            for (int c8 = half; c8 < nchH; c8 += kHalves, ++i) {
                float u[8], b[8], dyv[8];
                tmem_ld8(tmem_addr(tY, qtr, 8 * c8), u);
                ld8s(cv.c2 + 8 * c8, b);
                ld8<VEC>(drw, 8 * c8, valid ? H : 0, dyv);
                const uint32_t kb = th16 ? keep8(key3, th16, grow, H8, c8) : 0xffu;
                keepbits |= (unsigned long long)kb << (8 * i);
                tmem_wait_ld();
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    float yv = u[j] + b[j];
                    yv = (kb >> j) & 1u ? yv * dr.scale : 0.0f;
                    yv = (valid && 8 * c8 + j < H) ? yv : 0.0f;
                    ssum += yv;
                    dgate = fmaf(dyv[j], yv, dgate);
                }
            }
            row_exchange(cv.ex, half, prow, ssum, dgate);
            float gate = 1.0f, dsq = 0.0f;
            if (rr > 0) {
                const float sq = ssum / (float)H;
                const SeOut se = se_excite(sq, t, seq_base, T, rr, cv.se1, cv.se2);
                gate = se.gate;
                const float dq = valid ? dgate * gate * (1.0f - gate) : 0.0f;
                float da[kMaxRR];
#pragma unroll
                for (int k = 0; k < kMaxRR; ++k) da[k] = 0.0f;
                for (int tt = 0; tt < T; ++tt) {
                    const float dqt = __shfl_sync(0xffffffffu, dq, seq_base + tt);
#pragma unroll
                    for (int k = 0; k < kMaxRR; ++k)
                        if (k < rr) da[k] = fmaf(dqt, cv.se2[tt * rr + k], da[k]);
                }
#pragma unroll
                for (int k = 0; k < kMaxRR; ++k)
                    if (k < rr) {
                        const float dz = se.z[k] > 0.0f ? da[k] : 0.0f;
                        dsq = fmaf(dz, cv.se1[k * T + t], dsq);
                        if (valid && half == 0) {
                            gS2[k] = fmaf(dq, fmaxf(se.z[k], 0.0f), gS2[k]);
                            gS1[k] = fmaf(dz, sq, gS1[k]);
                        }
                    }
                dsq /= (float)H;
            }
            // dY2 = reg2'( dy * gate + dsq )
            i = 0;
#pragma unroll 1
            for (int c8 = half; c8 < NCH; c8 += kHalves, ++i) {
                float dyv[8];
                ld8<VEC>(drw, 8 * c8, valid ? H : 0, dyv);
                const uint32_t kb = (uint32_t)(keepbits >> (8 * i)) & 0xffu;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    float d = fmaf(dyv[j], gate, dsq);
                    d = (kb >> j) & 1u ? d * dr.scale : 0.0f;
                    dyv[j] = (valid && 8 * c8 + j < H) ? d : 0.0f;
                }
                put_chunk(bufX, P::PLANE, P::PS, prow, c8, dyv);
            }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            // dG2 = dY2 W2          (A = X K-major, B = W2 [H rows][ch cols] read MN-major: K = h)
            gemm3<0, 1>(tY, xB, xB + P::PLANE, P::PS, w2B, w2B + P::WPLANE, P::WPS, KP, KP / 16, false);
            // dW2[h][c] += sum_r dY2[r][h] G2[r][c]   (both MN-major, K = the 128 rows); column ch of G2 is all ones -> db2
            gemm3<1, 1>(tDW2, xB, xB + P::PLANE, P::PS, yB, yB + P::PLANE, P::PS, KP, 128 / 16, !first);
            mma_commit(&bars[1]);
        }
        // ---------------- E3: dU2 = dG2 * (reg1' act')(stored in TMEM by E1) -> operand Y; xhat -> operand X again
        mbar_wait(&bars[1], ph_mma, abortf);
        ph_mma ^= 1;
        tc_fence_after();
#pragma unroll 1
        for (int c8 = half; c8 < NCH; c8 += kHalves) {
            float u[8], dg[8], xh[8];
            tmem_ld8(tmem_addr(tU, qtr, 8 * c8), u);          // reg1' * act' (stored by E1)
            tmem_ld8(tmem_addr(tY, qtr, 8 * c8), dg);
            tmem_ld8(tmem_addr(tXH, qtr, 8 * c8), xh);
            tmem_wait_ld();
#pragma unroll
            for (int j = 0; j < 8; ++j) u[j] *= dg[j];
            put_chunk(bufY, P::PLANE, P::PS, prow, c8, u);
            put_chunk(bufX, P::PLANE, P::PS, prow, c8, xh);
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            // d xhat = dU2 W1'      (A = Y K-major, B = W1' [ch rows][H cols] read MN-major: K = c)
            gemm3<0, 1>(tU, yB, yB + P::PLANE, P::PS, w1B, w1B + P::WPLANE, P::WPS, KP, KP / 16, false);
            // Wt[c][h] += sum_r dU2[r][c] xhat[r][h]; column H of xhat is all ones -> db1'
            gemm3<1, 1>(tDW1, yB, yB + P::PLANE, P::PS, xB, xB + P::PLANE, P::PS, KP, 128 / 16, !first);
            mma_commit(&bars[1]);
        }
        first = false;
        // ---------------- E4: LayerNorm backward + residual -> staged dx1 row
        mbar_wait(&bars[1], ph_mma, abortf);
        ph_mma ^= 1;
        tc_fence_after();
        {
            float m1 = 0.0f, m2 = 0.0f;
#pragma unroll 1
            for (int c8 = half; c8 < nchH; c8 += kHalves) {
                float u[8], xh[8];
                tmem_ld8(tmem_addr(tU, qtr, 8 * c8), u);
                tmem_ld8(tmem_addr(tXH, qtr, 8 * c8), xh);
                tmem_wait_ld();
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float dv = 8 * c8 + j < H ? u[j] : 0.0f;
                    m1 += dv;
                    m2 = fmaf(dv, xh[j], m2);
                }
            }
            row_exchange(cv.ex, half, prow, m1, m2);
            m1 /= (float)H;
            m2 /= (float)H;
            float* orow = reinterpret_cast<float*>(bufX) + (size_t)drow * g.pitch;
#pragma unroll 1
            for (int c8 = half; c8 < nchH; c8 += kHalves) {
                float u[8], xh[8], dyv[8];
                tmem_ld8(tmem_addr(tU, qtr, 8 * c8), u);
                tmem_ld8(tmem_addr(tXH, qtr, 8 * c8), xh);
                ld8<VEC>(drw, 8 * c8, valid ? H : 0, dyv);
                tmem_wait_ld();
#pragma unroll
                for (int j = 0; j < 8; ++j) u[j] = fmaf(rstd, u[j] - m1 - xh[j] * m2, dyv[j]);
                if (valid) st8<VEC>(orow, 8 * c8, H, u);
            }
        }
        tc_fence_before();
        fence_async_smem();
        __syncthreads();
        if (warp == 0) {
            stage_out<VEC>(a.out, reinterpret_cast<const float*>(bufX), (size_t)tile * g.tile_rows, nrows, H, g.pitch, lane);
            if (next < ntiles) stage_in<VEC>(S2, a.dy, (size_t)next * g.tile_rows, tile_nrows(next), H, g.pitch, &bars[2], lane);
        }
    }
    if (warp == 0) bulk_wait_all0();
    __syncthreads();

    // ---------------- flush: Wt, dW2 (TMEM, lane = output row) -> global gradients
    // lane c (< ch) holds row c of Wt [ch][H | ones]; lane h (< H) holds row h of dW2 [H][ch | ones]
    if (!first) {
        float* stg = reinterpret_cast<float*>(bufX);          // [KP][KP+1] staging for lane-contiguous REDs
        constexpr int SP = KP + 1;
        tc_fence_after();
#pragma unroll 1
        for (int c8 = half; c8 < NCH; c8 += kHalves) {
            float u[8];
            tmem_ld8(tmem_addr(tDW1, qtr, 8 * c8), u);
            tmem_wait_ld();
            if (prow < KP)
#pragma unroll
                for (int j = 0; j < 8; ++j) stg[prow * SP + 8 * c8 + j] = u[j];
        }
        __syncthreads();
        for (int i = tid; i < ch * H; i += kCtaThreads) {
            const int c = i / H, h = i - c * H;
            red_add(a.g_w1 + i, stg[c * SP + h] * cv.gam[h]);
        }
        for (int h = tid; h < H; h += kCtaThreads) {
            float sg = 0.0f, sb = 0.0f;
#pragma unroll 8
            for (int c = 0; c < ch; ++c) {
                const float w = a.w1[(size_t)c * H + h];
                sg = fmaf(stg[c * SP + h], w, sg);
                sb = fmaf(stg[c * SP + H], w, sb);
            }
            red_add(a.g_ln_g + h, sg);
            red_add(a.g_ln_b + h, sb);
        }
        for (int c = tid; c < ch; c += kCtaThreads) red_add(a.g_b1 + c, stg[c * SP + H]);
        __syncthreads();
#pragma unroll 1
        for (int c8 = half; c8 < NCH; c8 += kHalves) {
            float u[8];
            tmem_ld8(tmem_addr(tDW2, qtr, 8 * c8), u);
            tmem_wait_ld();
            if (prow < KP)
#pragma unroll
                for (int j = 0; j < 8; ++j) stg[prow * SP + 8 * c8 + j] = u[j];
        }
        __syncthreads();
        for (int i = tid; i < H * ch; i += kCtaThreads) {
            const int h = i / ch, c = i - h * ch;
            red_add(a.g_w2 + i, stg[h * SP + c]);
        }
        for (int h = tid; h < H; h += kCtaThreads) red_add(a.g_b2 + h, stg[h * SP + ch]);
        if (rr > 0) {
            __syncthreads();
            float* acc = stg;                                  // [2][rr*T]
            for (int i = tid; i < 2 * rr * T; i += kCtaThreads) acc[i] = 0.0f;
            __syncthreads();
            if (lane_ok && half == 0)
                for (int k = 0; k < rr; ++k) {
                    atomicAdd(acc + k * T + t, gS1[k]);              // dS1[k][t]
                    atomicAdd(acc + rr * T + t * rr + k, gS2[k]);    // dS2[t][k]
                }
            __syncthreads();
            for (int i = tid; i < rr * T; i += kCtaThreads) {
                red_add(a.g_se1 + i, acc[i]);
                red_add(a.g_se2 + i, acc[rr * T + i]);
            }
        }
    }
    cta_end<TM_COLS>(abortf, a.abort_count, tmem, tid);
}

}  // namespace chan
}  // namespace mmx
