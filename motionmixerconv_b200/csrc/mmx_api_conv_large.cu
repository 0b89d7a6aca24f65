// ConvMixerBlock halves whose tile does not fit the fused kernels (mmx_conv.cuh keeps S whole sequences [C,T,E], their zero-padded
// copies and the conv weights in shared memory: C = 8, E = 192 with 5x9 ... 9x29 kernels -- most of the reference's Optuna grid,
// optuna_search/conv_optuna_main.py:339-342 -- needs > 227 KB), and BatchNorm halves with the max squeeze.  Same arithmetic,
//     y = x + SE(reg(act(conv2d(LN(x)))))          conv_mixer_model.py:129-142 (ConvBlock), :47-70 (MultiChanSELayer), :279-292
// as a chain of stage kernels with the intermediates in HBM, each tiled freely (the caller -- functional.ConvHalfLarge --
// sequences them; LayerNorm is mmx_ln_{fwd,bwd}, BatchNorm statistics mmx_bn1d_stats + mmx_bn_finalize / mmx_bn_coef):
//     forward :  n = LN(x)  ->  z = conv2d(n)  ->  [BN statistics of act(z)]  ->  y = x + SE(reg(act(z)))            (tail_fwd)
//     backward:  tail_bwd1 (SE backward: per-(b,t) gate, d squeeze, argmax; BN: sums of dR, dR*xhat)  ->  [mmx_bn_coef]
//                -> tail_bwd2 (dz)  ->  dn = conv2d(dz, flipped / transposed weights), dW, db (conv2d_wgrad)  ->  LN backward
// The convolutions are direct fp32 SIMT kernels: a CTA owns one sequence x one slab of EW embedding positions, stages the
// zero-padded input slab and all weights in shared memory, and every thread produces all output channels of 4 consecutive
// positions with a sliding register window (1 shared load per 4*C FMAs in the inner loop).
// Dropout masks are those of the fused kernels (dropout_quad on the global quad index: tests/masks_np.conv_masks is the twin).
#include "mmx_launch.cuh"

#if defined(MMX_HOST_EMU)
extern "C" int mmx_conv2d_large_fwd(const MmxConvHalfDesc*, int, const float*, const float*, const float*, float*, void*) {
    return fail(MMX_E_UNSUPPORTED, "mmx_conv2d_large_fwd: not in the emulator");
}
extern "C" int mmx_conv2d_large_wgrad(const MmxConvHalfDesc*, const float*, const float*, float*, float*, void*) {
    return fail(MMX_E_UNSUPPORTED, "mmx_conv2d_large_wgrad: not in the emulator");
}
extern "C" int mmx_conv_tail_fwd(const MmxConvHalfDesc*, const float*, const float*, const float*, const float*, const float*, float*, void*) {
    return fail(MMX_E_UNSUPPORTED, "mmx_conv_tail_fwd: not in the emulator");
}
extern "C" int mmx_conv_tail_bwd1(const MmxConvHalfDesc*, const float*, const float*, const float*, const float*, const float*, float*, float*, float*,
                                  double*, void*) {
    return fail(MMX_E_UNSUPPORTED, "mmx_conv_tail_bwd1: not in the emulator");
}
extern "C" int mmx_conv_tail_bwd2(const MmxConvHalfDesc*, const float*, const float*, const float*, const float*, const float*, float*, void*) {
    return fail(MMX_E_UNSUPPORTED, "mmx_conv_tail_bwd2: not in the emulator");
}
#else
using namespace mmx;

namespace {

constexpr int kLT = 256;          // threads per CTA
constexpr int kMaxTup = 12;       // weight-gradient tuples (ci, i, j) per thread

struct ConvL {
    int B, C, T, E, kt, kp, pt, pp;
    int EW, EWP, TP, netile;      // embedding positions per slab, padded slab width, padded rows, slabs per sequence
    int transposed;               // 0: w[co][ci][i][j] as is.  1: data gradient -- the kernel is read flipped and transposed
};

__device__ __forceinline__ float warp_sum_f(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// zero-padded input slab: dst[c][tt][ee] = src[b][c][tt - pt][e0 + ee - pp]
__device__ __forceinline__ void load_slab(float* dst, const float* src, const ConvL& d, int e0) {
    const int n = d.C * d.TP * d.EWP;
    for (int i = threadIdx.x; i < n; i += kLT) {
        const int ee = i % d.EWP, r = i / d.EWP, tt = r % d.TP, c = r / d.TP;
        const int t = tt - d.pt, e = e0 + ee - d.pp;
        dst[i] = (t >= 0 && t < d.T && e >= 0 && e < d.E) ? src[((size_t)c * d.T + t) * d.E + e] : 0.0f;
    }
}

// out[b][co][t][e] = bias[co] + sum_{ci,i,j} w[co][ci][i][j] in[b][ci][t + i - pt][e + j - pp]
template <int CO>
__global__ void __launch_bounds__(kLT) conv2d_fwd_kernel(const ConvL d, const float* __restrict__ in, const float* __restrict__ w,
                                                         const float* __restrict__ bias, float* __restrict__ out) {
    extern __shared__ float4 cl_smem[];
    float* w_s = reinterpret_cast<float*>(cl_smem);                 // [ci][i][j][CO]
    float* in_s = w_s + d.C * d.kt * d.kp * CO;                     // [ci][TP][EWP]
    const int C = d.C, kt = d.kt, kp = d.kp, ntap = C * kt * kp;
    for (int i = threadIdx.x; i < ntap * CO; i += kLT) {
        const int co = i % CO, tap = i / CO, j = tap % kp, ii = (tap / kp) % kt, ci = tap / (kp * kt);
        float v = 0.0f;
        if (co < C) v = d.transposed ? w[((size_t)(ci * C + co) * kt + (kt - 1 - ii)) * kp + (kp - 1 - j)] : w[((size_t)(co * C + ci) * kt + ii) * kp + j];
        w_s[i] = v;
    }
    const int e0 = blockIdx.x * d.EW, nq = d.EW / 4, nitems = d.T * nq;
    for (int b = blockIdx.y; b < d.B; b += gridDim.y) {
        __syncthreads();
        load_slab(in_s, in + (size_t)b * C * d.T * d.E, d, e0);
        __syncthreads();
        for (int item = threadIdx.x; item < nitems; item += kLT) {
            const int t = item / nq, q = item - t * nq;
            float acc[CO][4];
#pragma unroll
            for (int co = 0; co < CO; ++co) {
                const float bv = (bias && co < C) ? bias[co] : 0.0f;
                acc[co][0] = acc[co][1] = acc[co][2] = acc[co][3] = bv;
            }
            for (int ci = 0; ci < C; ++ci)
                for (int ii = 0; ii < kt; ++ii) {
                    const float* row = in_s + ((size_t)ci * d.TP + t + ii) * d.EWP + 4 * q;
                    const float* wr = w_s + (size_t)((ci * kt + ii) * kp) * CO;
                    float x0 = row[0], x1 = row[1], x2 = row[2], x3 = row[3];
                    for (int j = 0; j < kp; ++j) {
#pragma unroll
                        for (int co = 0; co < CO; ++co) {
                            const float wv = wr[j * CO + co];
                            acc[co][0] = fmaf(wv, x0, acc[co][0]);
                            acc[co][1] = fmaf(wv, x1, acc[co][1]);
                            acc[co][2] = fmaf(wv, x2, acc[co][2]);
                            acc[co][3] = fmaf(wv, x3, acc[co][3]);
                        }
                        x0 = x1; x1 = x2; x2 = x3; x3 = row[j + 4];       // EWP holds EW + kp + 3 columns
                    }
                }
#pragma unroll
            for (int co = 0; co < CO; ++co)
                if (co < C) {
                    float* o = out + (((size_t)b * C + co) * d.T + t) * d.E + e0 + 4 * q;
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (e0 + 4 * q + k < d.E) o[k] = acc[co][k];
                }
        }
    }
}

// dw[co][ci][i][j] += sum_{b,t,e} dz[b][co][t][e] n[b][ci][t + i - pt][e + j - pp];   db[co] += sum dz
template <int CO>
__global__ void __launch_bounds__(kLT) conv2d_wgrad_kernel(const ConvL d, const float* __restrict__ dz, const float* __restrict__ n, float* dw, float* db) {
    extern __shared__ float4 cl_smem[];
    float* dz_s = reinterpret_cast<float*>(cl_smem);                // [co][T][EW]
    float* n_s = dz_s + d.C * d.T * d.EW;                            // [ci][TP][EWP]
    __shared__ float db_s[8];
    const int C = d.C, kt = d.kt, kp = d.kp, ntap = C * kt * kp, T = d.T, EW = d.EW;
    if (threadIdx.x < 8) db_s[threadIdx.x] = 0.0f;
    float acc[kMaxTup][CO];
#pragma unroll
    for (int k = 0; k < kMaxTup; ++k)
#pragma unroll
        for (int co = 0; co < CO; ++co) acc[k][co] = 0.0f;
    const int e0 = blockIdx.x * EW;
    for (int b = blockIdx.y; b < d.B; b += gridDim.y) {
        __syncthreads();
        load_slab(n_s, n + (size_t)b * C * T * d.E, d, e0);
        for (int i = threadIdx.x; i < C * T * EW; i += kLT) {
            const int ee = i % EW, r = i / EW;
            dz_s[i] = e0 + ee < d.E ? dz[((size_t)b * C * T + r) * d.E + e0 + ee] : 0.0f;
        }
        __syncthreads();
        for (int co = 0; co < C; ++co) {
            float v = 0.0f;
            for (int i = threadIdx.x; i < T * EW; i += kLT) v += dz_s[co * T * EW + i];
            v = warp_sum_f(v);
            if ((threadIdx.x & 31) == 0) atomicAdd(db_s + co, v);
        }
#pragma unroll
        for (int k = 0; k < kMaxTup; ++k) {
            const int tap = threadIdx.x + k * kLT;
            if (tap < ntap) {
                const int j = tap % kp, ii = (tap / kp) % kt, ci = tap / (kp * kt);
                for (int t = 0; t < T; ++t) {
                    const float* nr = n_s + ((size_t)ci * d.TP + t + ii) * d.EWP + j;
                    const float* zr = dz_s + (size_t)t * EW;
                    for (int e = 0; e < EW; e += 4) {
                        const float n0 = nr[e], n1 = nr[e + 1], n2 = nr[e + 2], n3 = nr[e + 3];
#pragma unroll
                        for (int co = 0; co < CO; ++co)
                            if (co < C) {
                                const float4 z4 = *reinterpret_cast<const float4*>(zr + (size_t)co * T * EW + e);
                                acc[k][co] = fmaf(z4.x, n0, fmaf(z4.y, n1, fmaf(z4.z, n2, fmaf(z4.w, n3, acc[k][co]))));
                            }
                    }
                }
            }
        }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kMaxTup; ++k) {
        const int tap = threadIdx.x + k * kLT;
        if (tap < ntap) {
            const int j = tap % kp, ii = (tap / kp) % kt, ci = tap / (kp * kt);
#pragma unroll
            for (int co = 0; co < CO; ++co)
                if (co < C) atomicAdd(dw + ((size_t)(co * C + ci) * kt + ii) * kp + j, acc[k][co]);
        }
    }
    if (threadIdx.x < C) atomicAdd(db + threadIdx.x, db_s[threadIdx.x]);
}

// ------------------------------------------------------------------------------------------ tails
struct TailL {
    int B, C, T, E, rr, use_max, act, bn;     // bn: BatchNorm affine after the activation (else dropout, if any)
    uint32_t site;
    Dropout dr;
    const float *x, *z, *dy, *aff, *coef, *se1, *se2, *gd_in;
    float *y, *gd, *dz, *g_se1, *g_se2;
    double* sums;
};

// reg(act(z)) of the 4 elements of quad q of global row `grow` (+ act'(z) * reg' if da != nullptr)
template <int ACT>
__device__ __forceinline__ void quad_act(const TailL& a, const Dropout& dr, const float* zrow, size_t grow, int c, int q, float (&v)[4], float* da) {
    const int E = a.E, E4 = (E + 3) >> 2;
    float ks[4] = {1.0f, 1.0f, 1.0f, 1.0f};
    if (!a.bn && dr.thresh) dropout_quad(dr, a.site, (uint64_t)grow * E4 + q, ks);
    const float sc = a.bn ? a.aff[c] : 1.0f, sh = a.bn ? a.aff[a.C + c] : 0.0f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int e = 4 * q + k;
        float av = 0.0f, d = 0.0f;
        if (e < E) d = act_fwd_grad<ACT>(zrow[e], &av);
        v[k] = e < E ? (a.bn ? fmaf(av, sc, sh) : av * ks[k]) : 0.0f;
        if (da) da[k] = e < E ? d * (a.bn ? 1.0f : ks[k]) : 0.0f;
    }
}

// block-wide (value, index) arg-max / sum of per-thread partials; result valid in thread 0
__device__ __forceinline__ void block_reduce_pool(float& s, float& m, int& mi, float* red_f, int* red_i) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    s = warp_sum_f(s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float om = __shfl_xor_sync(0xffffffffu, m, o);
        const int oi = __shfl_xor_sync(0xffffffffu, mi, o);
        if (om > m || (om == m && oi < mi)) { m = om; mi = oi; }
    }
    __syncthreads();
    if (lane == 0) { red_f[wid] = s; red_f[8 + wid] = m; red_i[wid] = mi; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w2 = 1; w2 < kLT / 32; ++w2) {
            s += red_f[w2];
            if (red_f[8 + w2] > m || (red_f[8 + w2] == m && red_i[w2] < mi)) { m = red_f[8 + w2]; mi = red_i[w2]; }
        }
    }
}

// per-sequence forward statistics: pool[t] (mean or max over (c,e) of R = reg(act(z))), argmax, and with dy: dgate[t] = sum dy*R
template <int ACT>
__device__ __forceinline__ void seq_pool(const TailL& a, const Dropout& dr, int b, float* pool, int* amax, float* dgate, float* red_f, int* red_i) {
    const int C = a.C, T = a.T, E = a.E, E4 = (E + 3) >> 2;
    for (int t = 0; t < T; ++t) {
        float s = 0.0f, m = -INFINITY, dg = 0.0f;
        int mi = 0x7fffffff;
        for (int i = threadIdx.x; i < C * E4; i += kLT) {
            const int c = i / E4, q = i - c * E4;
            const size_t grow = ((size_t)b * C + c) * T + t;
            float v[4];
            quad_act<ACT>(a, dr, a.z + grow * E, grow, c, q, v, nullptr);
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (4 * q + k < E) {
                    s += v[k];
                    if (v[k] > m) { m = v[k]; mi = c * E + 4 * q + k; }
                    if (dgate) dg = fmaf(a.dy[grow * E + 4 * q + k], v[k], dg);
                }
        }
        float s2 = dg;
        block_reduce_pool(s, m, mi, red_f, red_i);
        if (threadIdx.x == 0) { pool[t] = a.use_max ? m : s / (float)(C * E); amax[t] = mi; }
        if (dgate) {
            int dummy_i = 0;
            float dummy_m = 0.0f;
            block_reduce_pool(s2, dummy_m, dummy_i, red_f, red_i);
            if (threadIdx.x == 0) dgate[t] = s2;
        }
    }
    __syncthreads();
}

__device__ __forceinline__ void se_gate(const TailL& a, const float* pool, float* zz, float* gate) {
    const int T = a.T, rr = a.rr;
    if (rr > 0) {
        if (threadIdx.x < rr) {
            float acc = 0.0f;
            for (int t = 0; t < T; ++t) acc = fmaf(a.se1[threadIdx.x * T + t], pool[t], acc);
            zz[threadIdx.x] = acc;
        }
        __syncthreads();
        if (threadIdx.x < T) {
            float q = 0.0f;
            for (int k = 0; k < rr; ++k) q = fmaf(a.se2[threadIdx.x * rr + k], fmaxf(zz[k], 0.0f), q);
            gate[threadIdx.x] = sigmoidf_(q);
        }
    } else if (threadIdx.x < T) {
        gate[threadIdx.x] = 1.0f;
    }
    __syncthreads();
}

constexpr int kMaxTS = 64;       // frames / SE width held in static shared arrays

template <int ACT>
__global__ void __launch_bounds__(kLT) tail_fwd_kernel(const TailL a) {
    __shared__ float pool[kMaxTS], gate[kMaxTS], zz[kMaxTS], red_f[16];
    __shared__ int amax[kMaxTS], red_i[8];
    const Dropout dr = resolve_dropout(a.dr);
    const int C = a.C, T = a.T, E = a.E, E4 = (E + 3) >> 2;
    for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
        if (a.rr > 0) {
            seq_pool<ACT>(a, dr, b, pool, amax, nullptr, red_f, red_i);
            se_gate(a, pool, zz, gate);
        }
        for (int i = threadIdx.x; i < C * T * E4; i += kLT) {
            const int q = i % E4, r = i / E4, t = r % T, c = r / T;
            const size_t grow = (size_t)b * C * T + r;
            float v[4];
            quad_act<ACT>(a, dr, a.z + grow * E, grow, c, q, v, nullptr);
            const float g = a.rr > 0 ? gate[t] : 1.0f;
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (4 * q + k < E) a.y[grow * E + 4 * q + k] = fmaf(v[k], g, a.x[grow * E + 4 * q + k]);
        }
        __syncthreads();
    }
}

// SE backward per sequence: gd[b][t] = (gate, d squeeze, argmax); SE weight gradients; BatchNorm: sums[c] += sum dR, sum dR*xhat
template <int ACT>
__global__ void __launch_bounds__(kLT) tail_bwd1_kernel(const TailL a) {
    __shared__ float pool[kMaxTS], gate[kMaxTS], zz[kMaxTS], dgate[kMaxTS], dq[kMaxTS], dzz[kMaxTS], ds[kMaxTS], red_f[16];
    __shared__ float gs1[kMaxTS * 8], gs2[kMaxTS * 8];
    __shared__ double bsum[16];
    __shared__ int amax[kMaxTS], red_i[8];
    const Dropout dr = resolve_dropout(a.dr);
    const int C = a.C, T = a.T, E = a.E, E4 = (E + 3) >> 2, rr = a.rr;
    for (int i = threadIdx.x; i < rr * T; i += kLT) { gs1[i] = 0.0f; gs2[i] = 0.0f; }
    if (threadIdx.x < 16) bsum[threadIdx.x] = 0.0;
    __syncthreads();
    for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
        if (rr > 0) {
            seq_pool<ACT>(a, dr, b, pool, amax, dgate, red_f, red_i);
            se_gate(a, pool, zz, gate);
            if (threadIdx.x < T) dq[threadIdx.x] = dgate[threadIdx.x] * gate[threadIdx.x] * (1.0f - gate[threadIdx.x]);
            __syncthreads();
            if (threadIdx.x < rr) {
                float da = 0.0f;
                for (int t = 0; t < T; ++t) da = fmaf(dq[t], a.se2[t * rr + threadIdx.x], da);
                dzz[threadIdx.x] = zz[threadIdx.x] > 0.0f ? da : 0.0f;
            }
            __syncthreads();
            if (threadIdx.x < T) {
                float acc = 0.0f;
                for (int k = 0; k < rr; ++k) acc = fmaf(dzz[k], a.se1[k * T + threadIdx.x], acc);
                ds[threadIdx.x] = acc;
            }
            for (int i = threadIdx.x; i < rr * T; i += kLT) {
                const int k = i / T, t = i - k * T;
                gs1[i] = fmaf(dzz[k], pool[t], gs1[i]);
                gs2[t * rr + k] = fmaf(dq[t], fmaxf(zz[k], 0.0f), gs2[t * rr + k]);
            }
            __syncthreads();
        }
        if (threadIdx.x < T) {
            float* g = a.gd + ((size_t)b * T + threadIdx.x) * 3;
            g[0] = rr > 0 ? gate[threadIdx.x] : 1.0f;
            g[1] = rr > 0 ? ds[threadIdx.x] : 0.0f;
            g[2] = rr > 0 ? (float)amax[threadIdx.x] : 0.0f;
        }
        if (a.bn) {
            for (int c = 0; c < C; ++c) {
                const float xs = a.aff[2 * C + c], xo = a.aff[3 * C + c];
                float s1 = 0.0f, s2 = 0.0f;
                for (int i = threadIdx.x; i < T * E4; i += kLT) {
                    const int t = i / E4, q = i - t * E4;
                    const size_t grow = ((size_t)b * C + c) * T + t;
                    const float g = rr > 0 ? gate[t] : 1.0f, dsv = rr > 0 ? ds[t] : 0.0f;
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const int e = 4 * q + k;
                        if (e < E) {
                            float av;
                            act_fwd_grad<ACT>(a.z[grow * E + e], &av);
                            float dR = a.dy[grow * E + e] * g;
                            if (rr > 0) dR += a.use_max ? (c * E + e == amax[t] ? dsv : 0.0f) : dsv / (float)(C * E);
                            s1 += dR;
                            s2 = fmaf(dR, fmaf(av, xs, xo), s2);
                        }
                    }
                }
                s1 = warp_sum_f(s1); s2 = warp_sum_f(s2);
                if ((threadIdx.x & 31) == 0) { atomicAdd(bsum + c, (double)s1); atomicAdd(bsum + 8 + c, (double)s2); }
            }
        }
        __syncthreads();
    }
    for (int i = threadIdx.x; i < rr * T; i += kLT) { atomicAdd(a.g_se1 + i, gs1[i]); atomicAdd(a.g_se2 + i, gs2[i]); }
    if (a.bn && threadIdx.x < C) { atomicAdd(a.sums + threadIdx.x, bsum[threadIdx.x]); atomicAdd(a.sums + C + threadIdx.x, bsum[8 + threadIdx.x]); }
}

// dz = d(loss)/d(conv output):  dR = dy*gate + d squeeze term;  dropout / identity: dz = dR * reg' * act'(z);
// BatchNorm: dz = k1*(dR - k2 - xhat*k3) * act'(z)
template <int ACT>
__global__ void __launch_bounds__(kLT) tail_bwd2_kernel(const TailL a) {
    const Dropout dr = resolve_dropout(a.dr);
    const int C = a.C, T = a.T, E = a.E, E4 = (E + 3) >> 2;
    const long long nquads = (long long)a.B * C * T * E4;
    for (long long i = (long long)blockIdx.x * kLT + threadIdx.x; i < nquads; i += (long long)gridDim.x * kLT) {
        const int q = (int)(i % E4);
        const size_t grow = (size_t)(i / E4);
        const int t = (int)(grow % T), c = (int)((grow / T) % C);
        const size_t b = grow / ((size_t)T * C);
        const float* g = a.gd_in + (b * T + t) * 3;
        const float gate = g[0], dsv = g[1];
        const int am = (int)g[2];
        float v[4], da[4];
        quad_act<ACT>(a, dr, a.z + grow * E, grow, c, q, v, da);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int e = 4 * q + k;
            if (e < E) {
                float dR = a.dy[grow * E + e] * gate;
                if (a.rr > 0) dR += a.use_max ? (c * E + e == am ? dsv : 0.0f) : dsv / (float)(C * E);
                float out;
                if (a.bn) {
                    // v = act*scale + shift  ->  xhat = act*xs + xo
                    float av;
                    act_fwd_grad<ACT>(a.z[grow * E + e], &av);
                    const float xh = fmaf(av, a.aff[2 * C + c], a.aff[3 * C + c]);
                    out = a.coef[c] * (dR - a.coef[C + c] - xh * a.coef[2 * C + c]) * da[k];
                } else {
                    out = dR * da[k];
                }
                a.dz[grow * E + e] = out;
            }
        }
    }
}

int plan_large(const MmxConvHalfDesc* d, bool wgrad, ConvL* out, size_t* smem, int* co) {
    if (!d) return fail(MMX_E_INVALID, "null descriptor");
    if (d->B <= 0 || d->C <= 0 || d->T <= 0 || d->E <= 0 || d->kt <= 0 || d->kp <= 0) return fail(MMX_E_INVALID, "non-positive dimension");
    if (d->C > 8) return fail(MMX_E_UNSUPPORTED, "conv_nChan %d > 8", d->C);
    if (d->pad_t < 0 || d->pad_p < 0 || d->pad_t > d->kt - 1 || d->pad_p > d->kp - 1)
        return fail(MMX_E_INVALID, "padding (%d,%d) does not keep the [T,E] shape for kernel (%d,%d)", d->pad_t, d->pad_p, d->kt, d->kp);
    const int CO = d->C <= 1 ? 1 : d->C <= 2 ? 2 : d->C <= 4 ? 4 : 8;
    if (wgrad && d->C * d->kt * d->kp > kMaxTup * kLT) return fail(MMX_E_UNSUPPORTED, "conv kernel %dx%dx(%d,%d): more than %d taps", d->C, d->C, d->kt, d->kp, kMaxTup * kLT);
    const DevInfo di = dev_info();
    ConvL m;
    m.B = d->B; m.C = d->C; m.T = d->T; m.E = d->E; m.kt = d->kt; m.kp = d->kp; m.pt = d->pad_t; m.pp = d->pad_p; m.transposed = 0;
    m.TP = d->T + d->kt - 1;
    auto bytes_of = [&](int EW) {
        const size_t slab = (size_t)m.C * m.TP * (EW + d->kp + 3);
        return (wgrad ? (size_t)m.C * m.T * EW + slab : (size_t)m.C * m.kt * m.kp * CO + slab) * 4 + 64;
    };
    const int EW = fit_tile(di, round_up(d->E, 4), 4, 4, true, bytes_of);
    if (EW) {
        m.EW = EW; m.EWP = EW + d->kp + 3; m.netile = (d->E + EW - 1) / EW;
        *out = m; *smem = bytes_of(EW); *co = CO;
        return MMX_OK;
    }
    return fail(MMX_E_UNSUPPORTED, "large ConvMixerBlock path: kernel %dx%dx(%d,%d) does not fit shared memory", d->C, d->C, d->kt, d->kp);
}

template <int CO>
int run_fwd(const ConvL& m, size_t smem, const float* in, const float* w, const float* bias, float* out, void* stream) {
    const DevInfo di = dev_info();
    int by = imax(1, (4 * di.sms + m.netile - 1) / m.netile);      // each CTA stages the weights once and loops over its sequences
    if (by > m.B) by = m.B;
    return launch_kernel(conv2d_fwd_kernel<CO>, dim3(m.netile, by), kLT, smem, stream, kNoPdl, m, in, w, bias, out);
}
template <int CO>
int run_wgrad(const ConvL& m, size_t smem, const float* dz, const float* n, float* dw, float* db, void* stream) {
    const DevInfo di = dev_info();
    int by = imax(1, (2 * di.sms + m.netile - 1) / m.netile);
    if (by > m.B) by = m.B;
    return launch_kernel(conv2d_wgrad_kernel<CO>, dim3(m.netile, by), kLT, smem, stream, kNoPdl, m, dz, n, dw, db);
}

int fill_tail(TailL& a, const MmxConvHalfDesc* d, const char* what) {
    if (!d) return fail(MMX_E_INVALID, "%s: null descriptor", what);
    if (d->B <= 0 || d->C <= 0 || d->C > 8 || d->T <= 0 || d->E <= 0) return fail(MMX_E_INVALID, "%s: bad sizes", what);
    if (d->act != MMX_ACT_GELU && d->act != MMX_ACT_MISH) return fail(MMX_E_INVALID, "Unknown activation function type: %d", d->act);
    if (d->T > kMaxTS || (d->use_se && (d->se_hidden < 1 || d->se_hidden > 8))) return fail(MMX_E_UNSUPPORTED, "%s: in_nTP %d / SE width %d", what, d->T, d->se_hidden);
    a = TailL();
    a.B = d->B; a.C = d->C; a.T = d->T; a.E = d->E; a.rr = d->use_se ? d->se_hidden : 0; a.use_max = d->use_max_pooling; a.act = d->act;
    a.site = (uint32_t)d->site;
    a.dr = make_dropout(d->dropout, d->training);
    return MMX_OK;
}

}  // namespace

// z = conv2d(in) (+ bias): the ConvBlock convolution (conv_mixer_model.py:133) when data_gradient == 0; with data_gradient != 0 the
// same kernel computes d(in) from d(z): weights read flipped and transposed, padding (k-1-pad), no bias.  in, out: [B,C,T,E].
extern "C" int mmx_conv2d_large_fwd(const MmxConvHalfDesc* d, int data_gradient, const float* in, const float* w, const float* bias, float* out,
                                    void* stream) {
    if (!in || !w || !out) return fail(MMX_E_INVALID, "mmx_conv2d_large_fwd: null tensor");
    ConvL m; size_t smem; int co;
    int rc = plan_large(d, false, &m, &smem, &co);
    if (rc) return rc;
    if (data_gradient) { m.transposed = 1; m.pt = d->kt - 1 - d->pad_t; m.pp = d->kp - 1 - d->pad_p; bias = nullptr; }
    switch (co) {
        case 1: return run_fwd<1>(m, smem, in, w, bias, out, stream);
        case 2: return run_fwd<2>(m, smem, in, w, bias, out, stream);
        case 4: return run_fwd<4>(m, smem, in, w, bias, out, stream);
        default: return run_fwd<8>(m, smem, in, w, bias, out, stream);
    }
}

// dw += dz (*) n, db += sum dz  (gradients of conv.weight [C,C,kt,kp] and conv.bias [C]); dz, n: [B,C,T,E]
extern "C" int mmx_conv2d_large_wgrad(const MmxConvHalfDesc* d, const float* dz, const float* n, float* dw, float* db, void* stream) {
    if (!dz || !n || !dw || !db) return fail(MMX_E_INVALID, "mmx_conv2d_large_wgrad: null tensor");
    ConvL m; size_t smem; int co;
    int rc = plan_large(d, true, &m, &smem, &co);
    if (rc) return rc;
    switch (co) {
        case 1: return run_wgrad<1>(m, smem, dz, n, dw, db, stream);
        case 2: return run_wgrad<2>(m, smem, dz, n, dw, db, stream);
        case 4: return run_wgrad<4>(m, smem, dz, n, dw, db, stream);
        default: return run_wgrad<8>(m, smem, dz, n, dw, db, stream);
    }
}

// y = x + SE(reg(act(z))): reg = dropout (d->dropout, training) or, bn_aff != null, the BatchNorm affine [scale|shift|..][C]
extern "C" int mmx_conv_tail_fwd(const MmxConvHalfDesc* d, const float* x, const float* z, const float* bn_aff, const float* se_w1,
                                 const float* se_w2, float* y, void* stream) {
    TailL a;
    int rc = fill_tail(a, d, "mmx_conv_tail_fwd");
    if (rc) return rc;
    if (!x || !z || !y || (a.rr > 0 && (!se_w1 || !se_w2))) return fail(MMX_E_INVALID, "mmx_conv_tail_fwd: null tensor");
    a.x = x; a.z = z; a.y = y; a.aff = bn_aff; a.bn = bn_aff != nullptr; a.se1 = se_w1; a.se2 = se_w2;
    const auto kern = a.act == MMX_ACT_GELU ? tail_fwd_kernel<ACT_GELU> : tail_fwd_kernel<ACT_MISH>;
    return launch_kernel(kern, capped_grid(dev_info(), a.B, 1, 8), kLT, 0, stream, kNoPdl, a);        // B >= 1: fill_tail
}

// SE backward: gd [B,T,3] = (gate, d squeeze, argmax); SE weight gradients accumulated; bn (4C vector) non-null: sums[0:C] += sum dR,
// sums[C:2C] += sum dR*xhat (then mmx_bn_coef)
extern "C" int mmx_conv_tail_bwd1(const MmxConvHalfDesc* d, const float* z, const float* dy, const float* bn, const float* se_w1,
                                  const float* se_w2, float* g_se_w1, float* g_se_w2, float* gd, double* sums, void* stream) {
    TailL a;
    int rc = fill_tail(a, d, "mmx_conv_tail_bwd1");
    if (rc) return rc;
    if (!z || !dy || !gd || (a.rr > 0 && (!se_w1 || !se_w2 || !g_se_w1 || !g_se_w2)) || (bn && !sums)) return fail(MMX_E_INVALID, "mmx_conv_tail_bwd1: null tensor");
    a.z = z; a.dy = dy; a.aff = bn; a.bn = bn != nullptr; a.se1 = se_w1; a.se2 = se_w2; a.g_se1 = g_se_w1; a.g_se2 = g_se_w2; a.gd = gd; a.sums = sums;
    const auto kern = a.act == MMX_ACT_GELU ? tail_bwd1_kernel<ACT_GELU> : tail_bwd1_kernel<ACT_MISH>;
    return launch_kernel(kern, capped_grid(dev_info(), a.B, 1, 4), kLT, 0, stream, kNoPdl, a);        // B >= 1: fill_tail
}

// dz [B,C,T,E] = gradient wrt the conv output from dy, gd (tail_bwd1) and, BatchNorm, bn + coef (mmx_bn_coef)
extern "C" int mmx_conv_tail_bwd2(const MmxConvHalfDesc* d, const float* z, const float* dy, const float* gd, const float* bn, const float* coef,
                                  float* dz, void* stream) {
    TailL a;
    int rc = fill_tail(a, d, "mmx_conv_tail_bwd2");
    if (rc) return rc;
    if (!z || !dy || !gd || !dz || ((bn != nullptr) != (coef != nullptr))) return fail(MMX_E_INVALID, "mmx_conv_tail_bwd2: null tensor");
    a.z = z; a.dy = dy; a.gd_in = gd; a.aff = bn; a.coef = coef; a.bn = bn != nullptr; a.dz = dz;
    const long long nquads = (long long)a.B * a.C * a.T * ((a.E + 3) / 4);
    const auto kern = a.act == MMX_ACT_GELU ? tail_bwd2_kernel<ACT_GELU> : tail_bwd2_kernel<ACT_MISH>;
    return launch_kernel(kern, capped_grid(dev_info(), nquads, kLT, 16), kLT, 0, stream, kNoPdl, a);
}
#endif
