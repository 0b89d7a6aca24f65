// The ConvBlock convolution of the large ConvMixer halves on the Blackwell tensor cores (tcgen05 + TMEM), sm_100a:
//
//     fwd   : out[b][co][t][e] = bias[co] + sum_{ci,i,j} w[co][ci][i][j] in[b][ci][t + i - pt][e + j - pp]
//     wgrad : dw[co][ci][i][j] += sum_{b,t,e} dz[b][co][t][e] n[b][ci][t + i - pt][e + j - pp],   db[co] += sum dz
//
// the arithmetic of conv2d_fwd_kernel / conv2d_wgrad_kernel (mmx_api_conv_large.cu), with the bf16x3 toolkit of mmx_tc5.cuh.
// The data gradient is the forward with the weights read flipped and transposed and padding (k-1-pad), as there.
//
// Tiling.  A work item is one sequence b and one WINDOW of 128 padded embedding positions c -> e' = m0 + c (m0 = win * ST).  The
// item's zero-padded input slab is staged once and split into hi / lo once per element, in the 16-bit panel layout with
//     rows  = (time tt, channel ci) -> slab row tt * C + ci          cols = the 128 window positions
// so for a fixed output frame t the taps (i, ci) are the CONTIGUOUS slab rows t*C + (i*C + ci): the slab is a GEMM operand at
// every t by moving the descriptor's start row, and nothing is copied per tap (no im2col).  The embedding taps j go into N:
//     fwd   : P[c][(co, j)] = sum_{(i,ci)} S[t*C + i*C + ci][c] W[(co, j)][(i, ci)]       M = 128 positions (slab, MN-major)
//                                                                                         N = C * jp (jp = kp rounded up to 8)
//                                                                                         K = kt * C rounded up to 16
//             out[co][t][m0 + c] = sum_j P[c + j][(co, j)]   (the diagonal sum: TMEM -> shared memory -> fp32 adds)
//     wgrad : D[(co, j)][(i, ci)] += sum_c Z[(co, j)][c] S[t*C + i*C + ci][c],   Z[(co, j)][c] = dz[co][t][m0 + c - j]
//                                                                                         M = C * jp (<= 2 x 128), N = K above
//                                                                                         K = the 128 window positions
// A window serves ST = 128 - (kp - 1) (rounded down to 8) output positions; windows overlap by kp - 1 slab columns.  The taps
// beyond kt * C in the padded K range are real slab rows of later frames (or zeros) times zero weights / ignored accumulator
// columns.  D stays in TMEM over the CTA's whole persistent loop and is flushed once; db is summed in fp32 from the staged dz.
// The forward keeps two accumulators in TMEM so the MMAs of frame t + 1 run under the diagonal sums of frame t.
#pragma once
#include "mmx_tc5.cuh"

namespace mmx {
namespace ctc5 {

using namespace tc5;

struct ConvTc5Args {
    const float* in;     // fwd: conv input [B,C,T,E] (data gradient: d(out)); wgrad: n [B,C,T,E]
    const float* w;      // fwd: [C,C,kt,kp]
    const float* bias;   // fwd, nullable
    const float* dz;     // wgrad: [B,C,T,E]
    float* out;          // fwd: [B,C,T,E]
    float *dw, *db;      // wgrad, accumulated
    int B, C, T, E, kt, kp, pt, pp;
    int transposed;      // fwd: 1 = data gradient (weights flipped and transposed)
    int* abort_count;
};

struct ConvGeom {
    int jp, NP, Kp, R, ST, nwin, MR;   // taps j per channel (padded), N, K, slab rows, outputs per window, windows, wgrad M rows
};
MMX_HD ConvGeom conv_tc5_geom(int C, int T, int E, int kt, int kp) {
    ConvGeom g;
    g.jp = (kp + 7) / 8 * 8;
    g.NP = (C * g.jp + 15) / 16 * 16;
    g.Kp = (kt * C + 15) / 16 * 16;
    g.R = (T - 1) * C + g.Kp;
    g.ST = (128 - (kp - 1)) / 8 * 8;
    g.nwin = g.ST > 0 ? (E + g.ST - 1) / g.ST : 0;
    g.MR = (C * g.jp + 127) / 128 * 128;
    return g;
}

// shared-memory layout (byte offsets from the 1024-aligned base; total includes the alignment slack)
struct ConvSmem {
    uint32_t slab, w, stg, z, dzs, bars, total;
};
MMX_HD ConvSmem conv_tc5_smem(const ConvGeom& g, int C, bool wgrad) {
    ConvSmem m;
    uint32_t o = 0;
    m.slab = o; o += up128(2u * 16u * (uint32_t)g.R * 16u);                         // hi + lo planes, 16 column groups
    m.w = o; o += wgrad ? 0u : up128(2u * (uint32_t)(g.Kp / 8) * g.NP * 16u);        // W[(co,j)][(i,ci)], K-major
    m.stg = o; o += wgrad ? 0u : up128((uint32_t)kHalves * 128u * (g.jp + 1) * 4u);  // diagonal-sum staging, one per half
    m.z = o; o += wgrad ? up128(2u * 16u * (uint32_t)g.MR * 16u) : 0u;             // Z[(co,j)][c], K-major
    m.dzs = o; o += wgrad ? up128((uint32_t)C * 128u * 4u) : 0u;                   // dz of one frame, [C][128]
    m.bars = o; o += 64 * 4;                                                        // barriers, TMEM slot, abort flag
    m.total = o + 1024;
    return m;
}

MMX_D uint8_t* align1024(uint8_t* p) { return reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(p) + 1023) & ~(uintptr_t)1023); }

// the zero-padded slab of sequence `src` for the window starting at padded position m0, split into the panel layout:
// S[tt*C + ci][c] = src[ci][tt - pt][m0 + c - pp]
MMX_D void stage_slab(uint8_t* slab, uint32_t plane, uint32_t ps, const float* src, const ConvTc5Args& a, int R, int m0, int tid) {
    const int C = a.C, T = a.T, E = a.E;
    for (int idx = tid; idx < R * 16; idx += kCtaThreads) {
        const int r = idx >> 4, c8 = idx & 15, tt = r / C, ci = r - tt * C, trow = tt - a.pt;
        const int e0 = m0 + 8 * c8 - a.pp;
        float v[8];
        if (trow >= 0 && trow < T) {
            const float* row = src + ((size_t)ci * T + trow) * E;
#pragma unroll
            for (int k = 0; k < 8; ++k) v[k] = (e0 + k >= 0 && e0 + k < E) ? __ldg(row + e0 + k) : 0.0f;
        } else {
#pragma unroll
            for (int k = 0; k < 8; ++k) v[k] = 0.0f;
        }
        put_chunk(slab, plane, ps, r, c8, v);
    }
}

// ------------------------------------------------------------------------------------------ forward / data gradient
template <int TM_COLS>
__global__ void __launch_bounds__(kCtaThreads, 1) conv_tc5_fwd_kernel(const ConvTc5Args a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* sm = align1024(smem_raw);
    const int C = a.C, T = a.T, E = a.E, kt = a.kt, kp = a.kp;
    const ConvGeom g = conv_tc5_geom(C, T, E, kt, kp);
    const ConvSmem m = conv_tc5_smem(g, C, false);
    uint8_t* slab = sm + m.slab;
    uint8_t* wb = sm + m.w;
    uint64_t* bars = reinterpret_cast<uint64_t*>(sm + m.bars);
    uint32_t* tslot = reinterpret_cast<uint32_t*>(bars + 4);
    volatile int* abortf = reinterpret_cast<volatile int*>(tslot + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, qtr = warp & 3, half = warp >> 2;
    const int prow = qtr * 32 + lane;
    const int jp = g.jp, SP = jp + 1;
    float* stg = reinterpret_cast<float*>(sm + m.stg) + half * 128 * SP;
    const uint32_t PS = (uint32_t)g.R * 16u, SPL = 16u * PS, WPS = (uint32_t)g.NP * 16u, WPL = (uint32_t)(g.Kp / 8) * WPS;
    cta_begin<TM_COLS>(bars, 2, abortf, tslot, tid);
    pdl_launch_dependents();
    for (int i = tid; i < (int)(2 * WPL / 16); i += kCtaThreads) reinterpret_cast<uint4*>(wb)[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();
    // B[n = co*jp + j][k = i*C + ci] = w(co, ci, i, j)   (the parameters: no predecessor in the stream writes them)
    for (int idx = tid; idx < C * C * kt * kp; idx += kCtaThreads) {
        const int j = idx % kp, i = (idx / kp) % kt, ci = (idx / (kp * kt)) % C, co = idx / (kp * kt * C);
        const float v = a.transposed ? a.w[((size_t)(ci * C + co) * kt + (kt - 1 - i)) * kp + (kp - 1 - j)] : a.w[idx];
        const Split s = split1(v);
        const uint32_t off = panel_off(co * jp + j, i * C + ci, WPS);
        *reinterpret_cast<uint16_t*>(wb + off) = (uint16_t)s.hi;
        *reinterpret_cast<uint16_t*>(wb + WPL + off) = (uint16_t)s.lo;
    }
    pdl_wait();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tslot;
    const uint32_t sB = smem_u32(slab), wB = smem_u32(wb);
    const int nitems = a.B * g.nwin, nrounds = (C + kHalves - 1) / kHalves;
    uint32_t ph = 0;                                  // bit s: phase of bars[s]
    auto issue = [&](int t) {
        const uint32_t r0 = (uint32_t)(t * C) * 16u;
        gemm3<1, 0>(tmem + (uint32_t)((t & 1) * g.NP), sB + r0, sB + SPL + r0, PS, wB, wB + WPL, WPS, g.NP, g.Kp / 16, false);
        mma_commit(&bars[t & 1]);
    };
    for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
        const int b = item / g.nwin, m0 = (item - b * g.nwin) * g.ST;
        stage_slab(slab, SPL, PS, a.in + (size_t)b * C * T * E, a, g.R, m0, tid);
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (tid == 0) { tc_fence_after(); issue(0); }
        for (int t = 0; t < T; ++t) {
            if (tid == 0 && t + 1 < T) { tc_fence_after(); issue(t + 1); }   // the other accumulator: read out last iteration
            mbar_wait(&bars[t & 1], (ph >> (t & 1)) & 1u, abortf);
            ph ^= 1u << (t & 1);
            tc_fence_after();
            const uint32_t acc = tmem + (uint32_t)((t & 1) * g.NP);
            for (int rnd = 0; rnd < nrounds; ++rnd) {
                const int co = half + kHalves * rnd;
                if (co < C) {
#pragma unroll 1
                    for (int c8 = 0; c8 < jp / 8; ++c8) {
                        float u[8];
                        tmem_ld8(tmem_addr(acc, qtr, co * jp + 8 * c8), u);
                        tmem_wait_ld();
#pragma unroll
                        for (int k = 0; k < 8; ++k) stg[prow * SP + 8 * c8 + k] = u[k];
                    }
                }
                __syncthreads();
                const int e = m0 + prow;
                if (co < C && prow < g.ST && e < E) {
                    float s = 0.0f;
                    for (int j = 0; j < kp; ++j) s += stg[(prow + j) * SP + j];
                    if (a.bias) s += __ldg(a.bias + co);
                    a.out[(((size_t)b * C + co) * T + t) * E + e] = s;
                }
                if (rnd + 1 == nrounds) tc_fence_before();
                __syncthreads();
            }
        }
    }
    cta_end<TM_COLS>(abortf, a.abort_count, tmem, tid);
}

// ------------------------------------------------------------------------------------------ weight gradient
template <int TM_COLS>
__global__ void __launch_bounds__(kCtaThreads, 1) conv_tc5_wgrad_kernel(const ConvTc5Args a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* sm = align1024(smem_raw);
    const int C = a.C, T = a.T, E = a.E, kt = a.kt, kp = a.kp;
    const ConvGeom g = conv_tc5_geom(C, T, E, kt, kp);
    const ConvSmem m = conv_tc5_smem(g, C, true);
    uint8_t* slab = sm + m.slab;
    uint8_t* zb = sm + m.z;
    float* dzs = reinterpret_cast<float*>(sm + m.dzs);
    uint64_t* bars = reinterpret_cast<uint64_t*>(sm + m.bars);
    uint32_t* tslot = reinterpret_cast<uint32_t*>(bars + 4);
    volatile int* abortf = reinterpret_cast<volatile int*>(tslot + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, qtr = warp & 3, half = warp >> 2;
    const int prow = qtr * 32 + lane;
    const int jp = g.jp, MT = g.MR / 128;
    const uint32_t PS = (uint32_t)g.R * 16u, SPL = 16u * PS, ZPS = (uint32_t)g.MR * 16u, ZPL = 16u * ZPS;
    cta_begin<TM_COLS>(bars, 1, abortf, tslot, tid);
    pdl_launch_dependents();
    pdl_wait();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tslot;
    const uint32_t sB = smem_u32(slab), zB = smem_u32(zb);
    const int nitems = a.B * g.nwin;
    uint32_t ph = 0;
    bool first = true, pend = false;
    float dbacc[2] = {0.0f, 0.0f};                    // db of channel (tid + 512 q) / 128
    auto wait_mma = [&]() {
        if (pend) { mbar_wait(&bars[0], ph, abortf); ph ^= 1u; pend = false; }
    };
    for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
        const int b = item / g.nwin, m0 = (item - b * g.nwin) * g.ST;
        const int nout = min(g.ST, E - m0);           // output positions e = m0 + x, x < nout, of this window
        wait_mma();                                   // the slab and Z are read by the last item's MMAs
        stage_slab(slab, SPL, PS, a.in + (size_t)b * C * T * E, a, g.R, m0, tid);
        for (int t = 0; t < T; ++t) {
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int idx = tid + q * kCtaThreads, co = idx >> 7, x = idx & 127;
                if (co < C) {
                    const float v = x < nout ? __ldg(a.dz + (((size_t)b * C + co) * T + t) * E + m0 + x) : 0.0f;
                    dzs[idx] = v;
                    dbacc[q] += v;
                }
            }
            __syncthreads();
            wait_mma();
            for (int idx = tid; idx < g.MR * 16; idx += kCtaThreads) {
                const int r = idx >> 4, c8 = idx & 15, co = r / jp, j = r - co * jp;
                float v[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const int x = 8 * c8 + k - j;
                    v[k] = (co < C && j < kp && x >= 0) ? dzs[co * 128 + x] : 0.0f;
                }
                put_chunk(zb, ZPL, ZPS, r, c8, v);
            }
            fence_async_smem();
            tc_fence_before();
            __syncthreads();
            if (tid == 0) {
                tc_fence_after();
                const uint32_t r0 = (uint32_t)(t * C) * 16u;
                for (int mt = 0; mt < MT; ++mt)
                    gemm3<0, 0>(tmem + (uint32_t)(mt * g.Kp), zB + (uint32_t)mt * 2048u, zB + ZPL + (uint32_t)mt * 2048u, ZPS, sB + r0,
                                sB + SPL + r0, PS, g.Kp, 128 / 16, !first);
                mma_commit(&bars[0]);
            }
            first = false;
            pend = true;
        }
    }
    wait_mma();
    tc_fence_after();
    if (!first) {
        for (int mt = 0; mt < MT; ++mt) {
            const int r = mt * 128 + prow, co = r / jp, j = r - co * jp;
#pragma unroll 1
            for (int c8 = half; c8 < g.Kp / 8; c8 += kHalves) {
                float u[8];
                tmem_ld8(tmem_addr(tmem + (uint32_t)(mt * g.Kp), qtr, 8 * c8), u);
                tmem_wait_ld();
                if (co < C && j < kp)
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        const int n = 8 * c8 + k, i = n / C, ci = n - i * C;
                        if (n < kt * C) red_add(a.dw + ((size_t)(co * C + ci) * kt + i) * kp + j, u[k]);
                    }
            }
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int co = (tid + q * kCtaThreads) >> 7;        // one channel per warp
            if (co < C) {
                float s = dbacc[q];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                if (lane == 0) red_add(a.db + co, s);
            }
        }
    }
    cta_end<TM_COLS>(abortf, a.abort_count, tmem, tid);
}

}  // namespace ctc5
}  // namespace mmx
