// Channel half of a MixerBlock on the Blackwell tensor cores, WIDE variant: 80 <= max(H, ch) <= 128 (K4 / AMASS-shaped models, the
// H = 128 cells of the large-batch sweep).  Same algorithm, tile geometry, operand layout and dropout streams as
// mmx_chan_tc5.cuh (read its header first); what changes is where things live, because at 128 columns
//   * the two split weight matrices (2 x 64 KB) no longer fit shared memory next to the activation operands: a prep kernel
//     writes W1' = W1 * gamma2 and W2, already split into bf16 hi / lo planes in the panel layout, plus b1' = b1 + W1 beta2,
//     into a device workspace once per launch, and every CTA streams them through ONE 64 KB shared-memory slot with the
//     bulk-copy engine (W1 -> W2 -> W1 ... per tile; the copies overlap the epilogue phases, the slot is L2-resident traffic);
//   * the backward's five 128-column TMEM regions would need 640 columns: the U and Y regions are reused (act' overwrites U,
//     dG overwrites Y, d xhat overwrites U), xhat is not parked but re-derived (from x1 for the operand, from the operand's
//     hi + lo planes for the LayerNorm backward), which leaves U | Y | Wt | dW2 = 512 columns exactly;
//   * there is no spare operand column for the ones that carry the bias gradients: db1', db2 are column sums of dU / dY2 over
//     the tile's rows, reduced by a recursive-halving shuffle (9 shuffles per 8-column chunk) into shared memory;
//   * the backward has no fp32 staging tiles: the x1 tile lands in the (then free) Y operand region, dy rows are read from
//     global memory by the row's threads (whole 32-byte sectors), dx1 rows are written the same way.
#pragma once
#include "mmx_chan_tc5.cuh"

namespace mmx {
namespace chanw {

using namespace tc5;
using namespace chan;

constexpr int KPW = 128;                                    // widest operand served
constexpr uint32_t kWsBytes = 2 * Panels<KPW>::WBUF + KPW * 4;    // workspace: W1' planes | W2 planes | b1' (any KP <= KPW)

// shared-memory layout (byte offsets from the 1024-aligned base; total includes the alignment slack)
struct WideSmem {
    uint32_t x, y, slot, s, small, total;
};
template <int KP>
MMX_HD WideSmem wide_smem(const Geo& g, bool bwd) {
    using P = Panels<KP>;
    const uint32_t st = stage_bytes(g), buf = umax(P::BUF, st);
    WideSmem m;
    uint32_t o = 0;
    m.x = o; o += buf;
    m.y = bwd ? o : m.x; o += bwd ? buf : 0;
    m.slot = o; o += P::WBUF;
    m.s = bwd ? m.y : o; o += bwd ? 0 : st;                         // backward: the x1 tile lands in the Y region
    m.small = o; o += (6 * KP + 2 * 32 * kMaxRR + 4 * kHalves * 128 + 64) * 4;   // c1f, c2, gamma2, db1, db2, spare | se1, se2 | exchange | barriers
    m.total = o + 1024;
    return m;
}

template <int KP>
struct CarveW {
    uint8_t *bufX, *bufY, *slot;
    float *S, *c1f, *c2, *gam, *db1, *db2, *se1, *se2, *ex;
    uint64_t* bars;
    uint32_t* tslot;
    volatile int* abortf;
    MMX_D CarveW(uint8_t* raw, const Geo& g, bool bwd) {
        uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~(uintptr_t)1023);
        const WideSmem m = wide_smem<KP>(g, bwd);
        bufX = sm + m.x;
        bufY = sm + m.y;
        slot = sm + m.slot;
        S = reinterpret_cast<float*>(sm + m.s);
        c1f = reinterpret_cast<float*>(sm + m.small);
        c2 = c1f + KP;
        gam = c2 + KP;
        db1 = gam + KP;
        db2 = db1 + KP;
        se1 = db2 + 2 * KP;
        se2 = se1 + 32 * kMaxRR;
        ex = se2 + 32 * kMaxRR;
        bars = reinterpret_cast<uint64_t*>(ex + 4 * kHalves * 128);
        tslot = reinterpret_cast<uint32_t*>(bars + 4);
        abortf = reinterpret_cast<volatile int*>(tslot + 1);
    }
};

// ------------------------------------------------------------------------------------------ weight preparation
// ws: W1' (hi plane, lo plane) | W2 (hi, lo) | b1'   -- panel layout, KPW x KPW, zero padded
template <int KPW>
static __global__ void __launch_bounds__(256) chan_prep_kernel(const ChanArgs a, uint8_t* ws) {
    using PW = Panels<KPW>;
    pdl_launch_dependents();
    pdl_wait();                // the previous kernel in the stream may still be reading the workspace
    const int H = a.H, ch = a.ch;
    const int gt = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
    for (int i = gt; i < KPW * KPW / 2; i += nt) {
        const int e = 2 * i, r = e / KPW, c = e - r * KPW;
        const uint32_t off = panel_off(r, c, PW::WPS);
        float2 v = make_float2(0.0f, 0.0f);
        if (r < ch && c < H) {
            v = *reinterpret_cast<const float2*>(a.w1 + (size_t)r * H + c);
            v.x *= a.ln_g[c];
            v.y *= a.ln_g[c + 1];
        }
        Split sp = split2(v.x, v.y);
        *reinterpret_cast<uint32_t*>(ws + off) = sp.hi;
        *reinterpret_cast<uint32_t*>(ws + PW::WPLANE + off) = sp.lo;
        v = make_float2(0.0f, 0.0f);
        if (r < H && c < ch) v = *reinterpret_cast<const float2*>(a.w2 + (size_t)r * ch + c);
        sp = split2(v.x, v.y);
        *reinterpret_cast<uint32_t*>(ws + PW::WBUF + off) = sp.hi;
        *reinterpret_cast<uint32_t*>(ws + PW::WBUF + PW::WPLANE + off) = sp.lo;
    }
    float* c1f = reinterpret_cast<float*>(ws + 2 * PW::WBUF);
    const int warp = gt >> 5, lane = gt & 31, nw = nt >> 5;
    for (int c = warp; c < KPW; c += nw) {
        float s = 0.0f;
        if (c < ch)
            for (int h = lane; h < H; h += 32) s = fmaf(a.w1[(size_t)c * H + h], a.ln_b[h], s);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) c1f[c] = c < ch ? s + a.b1[c] : 0.0f;
    }
}

// per-CTA constants that do not depend on the workspace.  Contains a CTA barrier.
template <int KPW>
MMX_D void small_params(const ChanArgs& a, const CarveW<KPW>& cv, int tid) {
    const int H = a.H, T = a.T, rr = a.rr;
    for (int c = tid; c < KPW; c += kCtaThreads) {
        cv.c2[c] = c < H ? a.b2[c] : 0.0f;
        cv.gam[c] = c < H ? a.ln_g[c] : 0.0f;
        cv.db1[c] = 0.0f;
        cv.db2[c] = 0.0f;
    }
    for (int i = tid; i < 32 * kMaxRR; i += kCtaThreads) {
        cv.se1[i] = (rr > 0 && i < rr * T) ? a.se1[i] : 0.0f;
        cv.se2[i] = (rr > 0 && i < rr * T) ? a.se2[i] : 0.0f;
    }
    __syncthreads();
}

template <int KPW>
MMX_D void load_weight(uint8_t* slot, const uint8_t* ws, int which, uint64_t* bar) {   // one thread
    mbar_expect_tx(bar, Panels<KPW>::WBUF);
    bulk_g2s(slot, ws + (size_t)which * Panels<KPW>::WBUF, Panels<KPW>::WBUF, bar);
}

// column sums over the warp's 32 rows of an 8-column chunk: lanes with (lane & 3) == 0 return the total of column
// 4*bit4 + 2*bit3 + bit2 of their lane index (recursive halving: 4 + 2 + 1 + 1 + 1 shuffles)
MMX_D float col_reduce8(const float (&v)[8], int lane) {
    float t4[4], t2[2];
    const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float keep = b4 ? v[j + 4] : v[j], send = b4 ? v[j] : v[j + 4];
        t4[j] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const float keep = b3 ? t4[j + 2] : t4[j], send = b3 ? t4[j] : t4[j + 2];
        t2[j] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
    const float keep = b2 ? t2[1] : t2[0], send = b2 ? t2[0] : t2[1];
    float t1 = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    t1 += __shfl_xor_sync(0xffffffffu, t1, 2);
    t1 += __shfl_xor_sync(0xffffffffu, t1, 1);
    return t1;
}
MMX_D void col_accumulate(float* dst, int c8, const float (&v)[8], int lane) {
    const float t = col_reduce8(v, lane);
    if ((lane & 3) == 0) atomicAdd(dst + 8 * c8 + ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1), t);
}

// xhat chunk from the operand's hi + lo planes (|error| <= 2^-17 |xhat|)
template <int KPW>
MMX_D void xhat_from_planes(const uint8_t* buf, int row, int c8, float (&xh)[8]) {
    using PW = Panels<KPW>;
    const uint4 h = *reinterpret_cast<const uint4*>(buf + c8 * PW::PS + row * 16);
    const uint4 l = *reinterpret_cast<const uint4*>(buf + PW::PLANE + c8 * PW::PS + row * 16);
    const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        xh[2 * i] = __uint_as_float(hw[i] << 16) + __uint_as_float(lw[i] << 16);
        xh[2 * i + 1] = __uint_as_float(hw[i] & 0xffff0000u) + __uint_as_float(lw[i] & 0xffff0000u);
    }
}

// ==========================================================================================
// forward
// ==========================================================================================
template <int ACT, int VEC, int KP>
__global__ void __launch_bounds__(kCtaThreads, KP <= 64 ? 2 : 1) chan_wide_fwd_kernel(const ChanArgs a, const uint8_t* ws) {
    using P = Panels<KP>;
    extern __shared__ uint8_t smem_raw[];
    const Geo g = make_geo(a.T, a.H, VEC);
    const CarveW<KP> cv(smem_raw, g, false);
    uint8_t* bufX = cv.bufX;
    float* S = cv.S;
    uint64_t* bars = cv.bars;
    volatile int* abortf = cv.abortf;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, qtr = warp & 3, half = warp >> 2;
    const int prow = qtr * 32 + lane;
    const int H = a.H, ch = a.ch, T = a.T, rr = a.rr;
    const Dropout dr = resolve_dropout(a.dr);
    const uint32_t th16 = dr.thresh >> 16;
    const uint32_t key2 = drop_key(dr.seed_lo, dr.seed_hi, a.site_base + 2, dr.step), key3 = drop_key(dr.seed_lo, dr.seed_hi, a.site_base + 3, dr.step);
    constexpr int TM_COLS = 4 * KP;      // U | Y | (residual rows resp. Wt) | dW2
    static_assert(TM_COLS == 256 || TM_COLS == 512, "KP = 64 or 128");
    constexpr int NCH = KP / 8;

    cta_begin<TM_COLS>(bars, 3, abortf, cv.tslot, tid);   // bars: x1 tile landed | MMA group done | weight slot landed
    pdl_launch_dependents();
    const int ntiles = (a.B + g.seq_per_tile - 1) / g.seq_per_tile;
    auto tile_nrows = [&](int tile) { return min(g.seq_per_tile, a.B - tile * g.seq_per_tile) * a.T; };
    small_params(a, cv, tid);
    pdl_wait();                // the prep kernel (and everything before it) has completed: workspace and x1 are readable
    for (int c = tid; c < KP; c += kCtaThreads) cv.c1f[c] = reinterpret_cast<const float*>(ws + 2 * P::WBUF)[c];
    uint32_t ph_w = 0;
    if ((int)blockIdx.x < ntiles) {
        if (tid == 0) load_weight<KP>(cv.slot, ws, 0, &bars[2]);
        if (warp == 0) stage_in<VEC>(S, a.x1, (size_t)blockIdx.x * g.tile_rows, tile_nrows(blockIdx.x), a.H, g.pitch, &bars[0], lane);
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *cv.tslot;
    const uint32_t tU = tmem, tY = tmem + KP, tXR = tmem + 2 * KP;
    const uint32_t xB = smem_u32(bufX), wB = smem_u32(cv.slot);

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
        const int next = tile + gridDim.x;

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
        if (warp == 0 && next < ntiles) stage_in<VEC>(S, a.x1, (size_t)next * g.tile_rows, tile_nrows(next), H, g.pitch, &bars[0], lane);
        if (tid == 0) {
            mbar_wait(&bars[2], ph_w, abortf);         // W1' in the slot
            ph_w ^= 1;
            tc_fence_after();
            gemm3<0, 0>(tU, xB, xB + P::PLANE, P::PS, wB, wB + P::WPLANE, P::WPS, KP, KP / 16, false);
            mma_commit(&bars[1]);
        }
        // ---------------- E1: U -> G = reg1(act(U + b1')) -> operand X; W2 streams into the slot meanwhile
        mbar_wait(&bars[1], ph_mma, abortf);
        ph_mma ^= 1;
        tc_fence_after();
        if (tid == 0) load_weight<KP>(cv.slot, ws, 1, &bars[2]);
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
            mbar_wait(&bars[2], ph_w, abortf);         // W2 in the slot
            ph_w ^= 1;
            tc_fence_after();
            gemm3<0, 0>(tY, xB, xB + P::PLANE, P::PS, wB, wB + P::WPLANE, P::WPS, KP, KP / 16, false);
            mma_commit(&bars[1]);
        }
        // ---------------- E2: Y2 -> reg2 -> SE -> + residual -> staged output row; W1' streams back for the next tile
        mbar_wait(&bars[1], ph_mma, abortf);
        ph_mma ^= 1;
        tc_fence_after();
        if (tid == 0 && next < ntiles) load_weight<KP>(cv.slot, ws, 0, &bars[2]);
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
template <int ACT, int VEC, int KP>
__global__ void __launch_bounds__(kCtaThreads, KP <= 64 ? 2 : 1) chan_wide_bwd_kernel(const ChanArgs a, const uint8_t* ws) {
    using P = Panels<KP>;
    extern __shared__ uint8_t smem_raw[];
    const Geo g = make_geo(a.T, a.H, VEC);
    const CarveW<KP> cv(smem_raw, g, true);
    uint8_t* bufX = cv.bufX;                  // xhat -> dY2 -> xhat again
    uint8_t* bufY = cv.bufY;                  // x1 tile (fp32) -> G2 -> dU2
    float* S1 = cv.S;
    uint64_t* bars = cv.bars;
    volatile int* abortf = cv.abortf;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, qtr = warp & 3, half = warp >> 2;
    const int prow = qtr * 32 + lane;
    const int H = a.H, ch = a.ch, T = a.T, rr = a.rr;
    const Dropout dr = resolve_dropout(a.dr);
    const uint32_t th16 = dr.thresh >> 16;
    const uint32_t key2 = drop_key(dr.seed_lo, dr.seed_hi, a.site_base + 2, dr.step), key3 = drop_key(dr.seed_lo, dr.seed_hi, a.site_base + 3, dr.step);
    constexpr int TM_COLS = 4 * KP;      // U | Y | Wt | dW2
    static_assert(TM_COLS == 256 || TM_COLS == 512, "KP = 64 or 128");
    constexpr int NCH = KP / 8;
    constexpr int CPT = NCH / kHalves;        // chunks per thread and pass

    cta_begin<TM_COLS>(bars, 3, abortf, cv.tslot, tid);   // bars: x1 tile landed | MMA group done | weight slot landed
    pdl_launch_dependents();
    const int ntiles = (a.B + g.seq_per_tile - 1) / g.seq_per_tile;
    auto tile_nrows = [&](int tile) { return min(g.seq_per_tile, a.B - tile * g.seq_per_tile) * a.T; };
    small_params(a, cv, tid);
    pdl_wait();
    for (int c = tid; c < KP; c += kCtaThreads) cv.c1f[c] = reinterpret_cast<const float*>(ws + 2 * P::WBUF)[c];
    uint32_t ph_w = 0;
    if ((int)blockIdx.x < ntiles) {
        if (tid == 0) load_weight<KP>(cv.slot, ws, 0, &bars[2]);
        if (warp == 0) stage_in<VEC>(S1, a.x1, (size_t)blockIdx.x * g.tile_rows, tile_nrows(blockIdx.x), a.H, g.pitch, &bars[0], lane);
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *cv.tslot;
    // U2 -> reg1' act' -> d xhat | Y2 -> dG2 | Wt = dU^T xhat | dW2
    const uint32_t tU = tmem, tY = tmem + KP, tDW1 = tmem + 2 * KP, tDW2 = tmem + 3 * KP;
    const uint32_t xB = smem_u32(bufX), yB = smem_u32(bufY), wB = smem_u32(cv.slot);

    const bool lane_ok = lane < g.rpw;
    const int t = lane_ok ? lane % T : 0;
    const int seq_base = lane_ok ? (lane / T) * T : 0;
    const int drow = qtr * g.rpw + (lane_ok ? lane : 0);
    const int nchH = (H + 7) >> 3;
    const uint32_t ch8 = (uint32_t)(ch + 7) >> 3, H8 = (uint32_t)nchH;
    uint32_t ph_x = 0, ph_mma = 0;
    bool first = true;
    float gS1[kMaxRR], gS2[kMaxRR];
#pragma unroll
    for (int k = 0; k < kMaxRR; ++k) gS1[k] = gS2[k] = 0.0f;

    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int nrows = tile_nrows(tile);
        const bool valid = lane_ok && drow < nrows;
        const size_t grow = (size_t)tile * g.tile_rows + drow;
        const int next = tile + gridDim.x;
        const float* srow = S1 + (size_t)drow * g.pitch;
        const float* xg = a.x1 + grow * H;          // the row in global memory (read again after the Y region is overwritten)
        const float* dyg = a.dy + grow * H;
        float* outg = a.out + grow * H;

        // ---------------- P0: xhat = LN2(x1) without affine -> operand X
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
            for (int j = 0; j < 8; ++j) v[j] = (valid && 8 * c8 + j < H) ? (v[j] - mean) * rstd : 0.0f;
            put_chunk(bufX, P::PLANE, P::PS, prow, c8, v);
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();   // operand X complete; the x1 tile (Y region) is consumed
        if (tid == 0) {
            if (first) {                               // later tiles: W1' was waited for by the previous tile's last product
                mbar_wait(&bars[2], ph_w, abortf);     // W1' in the slot
                ph_w ^= 1;
            }
            tc_fence_after();
            gemm3<0, 0>(tU, xB, xB + P::PLANE, P::PS, wB, wB + P::WPLANE, P::WPS, KP, KP / 16, false);
            mma_commit(&bars[1]);
        }
        // ---------------- E1: G2 = reg1(act(U2 + b1')) -> operand Y; TMEM keeps reg1'(.) * act'(U2 + b1') in place of U2
        mbar_wait(&bars[1], ph_mma, abortf);
        ph_mma ^= 1;
        tc_fence_after();
        if (tid == 0) load_weight<KP>(cv.slot, ws, 1, &bars[2]);
#pragma unroll 1
        for (int c8 = half; c8 < NCH; c8 += kHalves) {
            float u[8], b[8], dact[8];
            tmem_ld8(tmem_addr(tU, qtr, 8 * c8), u);
            ld8s(cv.c1f + 8 * c8, b);
            const uint32_t kb = th16 ? keep8(key2, th16, (uint32_t)grow, ch8, c8) : 0xffu;
            tmem_wait_ld();
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int c = 8 * c8 + j;
                float gv;
                const float da = act_fwd_grad<ACT>(u[j] + b[j], &gv);
                const float ks = (kb >> j) & 1u ? dr.scale : 0.0f;
                dact[j] = (valid && c < ch) ? da * ks : 0.0f;
                u[j] = (valid && c < ch) ? gv * ks : 0.0f;
            }
            put_chunk(bufY, P::PLANE, P::PS, prow, c8, u);
            tmem_st8(tmem_addr(tU, qtr, 8 * c8), dact);
        }
        tmem_wait_st();
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            mbar_wait(&bars[2], ph_w, abortf);         // W2 in the slot
            ph_w ^= 1;
            tc_fence_after();
            gemm3<0, 0>(tY, yB, yB + P::PLANE, P::PS, wB, wB + P::WPLANE, P::WPS, KP, KP / 16, false);
            mma_commit(&bars[1]);
        }
        // ---------------- E2: y2, SE forward + backward, dY2 -> operand X, db2
        float dyv[CPT][8];                             // the thread's chunks of the dy row (global reads in flight over the MMA wait)
#pragma unroll
        for (int i = 0; i < CPT; ++i) ld8<VEC>(dyg, 8 * (half + kHalves * i), valid ? H : 0, dyv[i]);
        mbar_wait(&bars[1], ph_mma, abortf);
        ph_mma ^= 1;
        tc_fence_after();
        {
            float ssum = 0.0f, dgate = 0.0f;
            uint32_t keepbits = 0u;
#pragma unroll
            for (int i = 0; i < CPT; ++i) {
                const int c8 = half + kHalves * i;
                float u[8], b[8];
                tmem_ld8(tmem_addr(tY, qtr, 8 * c8), u);
                ld8s(cv.c2 + 8 * c8, b);
                const uint32_t kb = th16 ? keep8(key3, th16, (uint32_t)grow, H8, c8) : 0xffu;
                keepbits |= kb << (8 * i);
                tmem_wait_ld();
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    float yv = u[j] + b[j];
                    yv = (kb >> j) & 1u ? yv * dr.scale : 0.0f;
                    yv = (valid && 8 * c8 + j < H) ? yv : 0.0f;
                    ssum += yv;
                    dgate = fmaf(dyv[i][j], yv, dgate);
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
#pragma unroll
            for (int i = 0; i < CPT; ++i) {
                const int c8 = half + kHalves * i;
                const uint32_t kb = (keepbits >> (8 * i)) & 0xffu;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    float d = fmaf(dyv[i][j], gate, dsq);
                    d = (kb >> j) & 1u ? d * dr.scale : 0.0f;
                    dyv[i][j] = (valid && 8 * c8 + j < H) ? d : 0.0f;
                }
                put_chunk(bufX, P::PLANE, P::PS, prow, c8, dyv[i]);
                col_accumulate(cv.db2, c8, dyv[i], lane);
            }
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            // dG2 = dY2 W2          (A = X K-major, B = W2 [H rows][ch cols] read MN-major: K = h)
            gemm3<0, 1>(tY, xB, xB + P::PLANE, P::PS, wB, wB + P::WPLANE, P::WPS, KP, KP / 16, false);
            // dW2[h][c] += sum_r dY2[r][h] G2[r][c]   (both MN-major, K = the 128 rows)
            gemm3<1, 1>(tDW2, xB, xB + P::PLANE, P::PS, yB, yB + P::PLANE, P::PS, KP, 128 / 16, !first);
            mma_commit(&bars[1]);
        }
        // ---------------- E3: dU2 = dG2 * (reg1' act') -> operand Y, db1'; xhat -> operand X again (from x1 in global memory)
        float xv[CPT][8];
#pragma unroll
        for (int i = 0; i < CPT; ++i) ld8<VEC>(xg, 8 * (half + kHalves * i), valid ? H : 0, xv[i]);
        mbar_wait(&bars[1], ph_mma, abortf);
        ph_mma ^= 1;
        tc_fence_after();
        if (tid == 0) load_weight<KP>(cv.slot, ws, 0, &bars[2]);
#pragma unroll
        for (int i = 0; i < CPT; ++i) {
            const int c8 = half + kHalves * i;
            float u[8], dg[8];
            tmem_ld8(tmem_addr(tU, qtr, 8 * c8), u);
            tmem_ld8(tmem_addr(tY, qtr, 8 * c8), dg);
            tmem_wait_ld();
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                u[j] *= dg[j];
                xv[i][j] = (valid && 8 * c8 + j < H) ? (xv[i][j] - mean) * rstd : 0.0f;
            }
            put_chunk(bufY, P::PLANE, P::PS, prow, c8, u);
            put_chunk(bufX, P::PLANE, P::PS, prow, c8, xv[i]);
            col_accumulate(cv.db1, c8, u, lane);
        }
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) {
            mbar_wait(&bars[2], ph_w, abortf);         // W1' in the slot (stays there for the next tile's first product)
            ph_w ^= 1;
            tc_fence_after();
            // d xhat = dU2 W1'      (A = Y K-major, B = W1' [ch rows][H cols] read MN-major: K = c)
            gemm3<0, 1>(tU, yB, yB + P::PLANE, P::PS, wB, wB + P::WPLANE, P::WPS, KP, KP / 16, false);
            // Wt[c][h] += sum_r dU2[r][c] xhat[r][h]
            gemm3<1, 1>(tDW1, yB, yB + P::PLANE, P::PS, xB, xB + P::PLANE, P::PS, KP, 128 / 16, !first);
            mma_commit(&bars[1]);
        }
        first = false;
        // ---------------- E4: LayerNorm backward + residual -> dx1 row (global)
#pragma unroll
        for (int i = 0; i < CPT; ++i) ld8<VEC>(dyg, 8 * (half + kHalves * i), valid ? H : 0, dyv[i]);
        mbar_wait(&bars[1], ph_mma, abortf);
        ph_mma ^= 1;
        tc_fence_after();
        if (warp == 0 && next < ntiles)                // the Y region is free: the next x1 tile lands there
            stage_in<VEC>(S1, a.x1, (size_t)next * g.tile_rows, tile_nrows(next), H, g.pitch, &bars[0], lane);
        {
            float m1 = 0.0f, m2 = 0.0f;
#pragma unroll
            for (int i = 0; i < CPT; ++i) {
                const int c8 = half + kHalves * i;
                float u[8];
                tmem_ld8(tmem_addr(tU, qtr, 8 * c8), u);
                xhat_from_planes<KP>(bufX, prow, c8, xv[i]);
                tmem_wait_ld();
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float dv = 8 * c8 + j < H ? u[j] : 0.0f;
                    m1 += dv;
                    m2 = fmaf(dv, xv[i][j], m2);
                }
            }
            row_exchange(cv.ex, half, prow, m1, m2);
            m1 /= (float)H;
            m2 /= (float)H;
#pragma unroll
            for (int i = 0; i < CPT; ++i) {
                const int c8 = half + kHalves * i;
                float u[8];
                tmem_ld8(tmem_addr(tU, qtr, 8 * c8), u);
                tmem_wait_ld();
#pragma unroll
                for (int j = 0; j < 8; ++j) u[j] = fmaf(rstd, u[j] - m1 - xv[i][j] * m2, dyv[i][j]);
                if (valid) st8<VEC>(outg, 8 * c8, H, u);
            }
        }
        tc_fence_before();
        __syncthreads();       // every thread is done with the X planes and the U region before the next tile overwrites them
    }
    __syncthreads();

    // ---------------- flush: Wt, dW2 (TMEM, lane = output row) -> global gradients
    if (!first) {
        float* stg = reinterpret_cast<float*>(bufX);          // [KP][KP], columns rotated by the row (conflict-free stores)
        tc_fence_after();
#pragma unroll 1
        for (int c8 = half; c8 < NCH; c8 += kHalves) {
            float u[8];
            tmem_ld8(tmem_addr(tDW1, qtr, 8 * c8), u);
            tmem_wait_ld();
            if (prow < KP)
#pragma unroll
                for (int j = 0; j < 8; ++j) stg[prow * KP + ((8 * c8 + j + prow) & (KP - 1))] = u[j];
        }
        __syncthreads();
        for (int i = tid; i < ch * H; i += kCtaThreads) {
            const int c = i / H, h = i - c * H;
            red_add(a.g_w1 + i, stg[c * KP + ((h + c) & (KP - 1))] * cv.gam[h]);
        }
        for (int h = tid; h < H; h += kCtaThreads) {
            float sg = 0.0f, sb = 0.0f;
#pragma unroll 8
            for (int c = 0; c < ch; ++c) {
                const float w = a.w1[(size_t)c * H + h];
                sg = fmaf(stg[c * KP + ((h + c) & (KP - 1))], w, sg);
                sb = fmaf(cv.db1[c], w, sb);
            }
            red_add(a.g_ln_g + h, sg);
            red_add(a.g_ln_b + h, sb);
        }
        for (int c = tid; c < ch; c += kCtaThreads) red_add(a.g_b1 + c, cv.db1[c]);
        __syncthreads();
#pragma unroll 1
        for (int c8 = half; c8 < NCH; c8 += kHalves) {
            float u[8];
            tmem_ld8(tmem_addr(tDW2, qtr, 8 * c8), u);
            tmem_wait_ld();
            if (prow < KP)
#pragma unroll
                for (int j = 0; j < 8; ++j) stg[prow * KP + ((8 * c8 + j + prow) & (KP - 1))] = u[j];
        }
        __syncthreads();
        for (int i = tid; i < H * ch; i += kCtaThreads) {
            const int h = i / ch, c = i - h * ch;
            red_add(a.g_w2 + i, stg[h * KP + ((c + h) & (KP - 1))]);
        }
        for (int h = tid; h < H; h += kCtaThreads) red_add(a.g_b2 + h, cv.db2[h]);
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

}  // namespace chanw
}  // namespace mmx
