// MlpMixer with regularization == -1: BatchNorm1d inside the MLP blocks (h36m/mlp_mixer.py:72-73 reg1/reg2 = BatchNorm1d(mlp_bn_dim),
// applied at :90-94).  Batch statistics are global over the batch, so a MixerBlock cannot be one kernel: it runs as a chain of
// stage kernels (the caller -- functional.MlpBnBlock -- sequences them; include/mmx.h documents the chain):
//
//     token half    LN1 (written transposed [B,H,T]) -> fc1 -> [stats] -> BN(act(.)) -> fc2 -> [stats] -> BN -> SE -> + x
//     channel half  LN2                              -> fc1 -> [stats] -> BN(act(.)) -> fc2 -> [stats] -> BN -> SE -> + x1
//
// token MLP:   tensors [B, H, *]: BatchNorm1d(hidden_dim) normalises every hidden column h over (batch, last dim)
// channel MLP: tensors [B, T, *]: BatchNorm1d(seq_len)    normalises every frame t over (batch, last dim)
// i.e. both are "[N, C, L] with statistics per c over (n, l)", one kernel family.  The fc layers are mmx_linear_{fwd,bwd}.
// The per-channel vectors are those of the ConvMixer BatchNorm path (mmx_bn_finalize / mmx_bn_coef):
//     bn   = [scale | shift | xs | xo][C]     R = a*scale + shift,  xhat = a*xs + xo          (a = act(u) or u)
//     coef = [k1 | k2 | k3][C]                dA = k1 * (dR - k2 - xhat*k3)
// fp32 CUDA-core kernels (a warp per row; the path is an Optuna option of the reference, optuna_search/optuna_main.py:189-190,
// not a benchmark configuration).
#include "mmx_launch.cuh"

#if defined(MMX_HOST_EMU)
#define MMX_BNMLP_STUB(name, ...) extern "C" int name(__VA_ARGS__) { return fail(MMX_E_UNSUPPORTED, #name ": not in the emulator"); }
MMX_BNMLP_STUB(mmx_ln_fwd, long long, int, int, const float*, const float*, const float*, float*, float*, void*)
MMX_BNMLP_STUB(mmx_ln_bwd, long long, int, int, const float*, const float*, const float*, const float*, const float*, float*, float*, float*, void*)
MMX_BNMLP_STUB(mmx_bn1d_stats, long long, int, int, int, const float*, double*, void*)
MMX_BNMLP_STUB(mmx_bn1d_apply, long long, int, int, int, const float*, const float*, float*, void*)
MMX_BNMLP_STUB(mmx_bn1d_bwd_reduce, long long, int, int, int, const float*, const float*, const float*, double*, void*)
MMX_BNMLP_STUB(mmx_bn1d_bwd_apply, long long, int, int, int, const float*, const float*, const float*, const float*, float*, void*)
MMX_BNMLP_STUB(mmx_se_res_fwd, int, int, int, int, int, int, int, const float*, const float*, const float*, const float*, const float*, float*, void*)
MMX_BNMLP_STUB(mmx_se_res_bwd, int, int, int, int, int, int, int, const float*, const float*, const float*, const float*, const float*, float*, float*, float*, void*)
#else
using namespace mmx;

namespace {

constexpr int kT = 256;
constexpr int ACT_ID = 2;

template <int ACT>
__device__ __forceinline__ float actf(float u) {
    if constexpr (ACT == ACT_ID) return u;
    else return act_fwd<ACT>(u);
}
template <int ACT>
__device__ __forceinline__ float actf_grad(float u, float* a) {
    if constexpr (ACT == ACT_ID) { *a = u; return 1.0f; }
    else return act_fwd_grad<ACT>(u, a);
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ------------------------------------------------------------------------------------------ LayerNorm over rows
// y = LN(x) * g + b, rows of width H; stats[r] = (mean, rstd).  Tt > 0: row r = (b, t) of a [B, Tt, H] tensor and the output is
// written transposed, y[b][h][t]  (MixerBlock.forward: y = self.LN1(x); y = y.transpose(1, 2), mlp_mixer.py:146-149).
__global__ void __launch_bounds__(kT) ln_fwd_kernel(const float* __restrict__ x, const float* __restrict__ g, const float* __restrict__ b,
                                                    float* __restrict__ y, float* __restrict__ stats, long long R, int H, int Tt) {
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarp = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long r = warp; r < R; r += nwarp) {
        const float* xr = x + r * H;
        const float c0 = xr[0];
        float s = 0.0f, ss = 0.0f;
        for (int h = lane; h < H; h += 32) { const float d = xr[h] - c0; s += d; ss = fmaf(d, d, ss); }
        s = warp_sum(s); ss = warp_sum(ss);
        const float ms = s / (float)H, mean = c0 + ms;
        const float rstd = 1.0f / sqrtf(fmaxf(ss / (float)H - ms * ms, 0.0f) + 1e-5f);
        if (lane == 0) { stats[2 * r] = mean; stats[2 * r + 1] = rstd; }
        const long long bb = Tt > 0 ? r / Tt : 0;
        const int t = Tt > 0 ? (int)(r - bb * Tt) : 0;
        for (int h = lane; h < H; h += 32) {
            const float v = fmaf((xr[h] - mean) * rstd, g[h], b[h]);
            if (Tt > 0) y[(bb * H + h) * Tt + t] = v; else y[r * H + h] = v;
        }
    }
}

// dx = res + LN backward(dy); dg += sum dy * xhat, db += sum dy.  Tt > 0: dy is laid out transposed ([B][H][Tt]).
__global__ void __launch_bounds__(kT) ln_bwd_kernel(const float* __restrict__ x, const float* __restrict__ stats, const float* __restrict__ g,
                                                    const float* __restrict__ dy, const float* res, float* dx, float* dg, float* db,
                                                    long long R, int H, int Tt) {
    extern __shared__ float ln_sm[];
    float* dgs = ln_sm;
    float* dbs = ln_sm + H;
    for (int h = threadIdx.x; h < 2 * H; h += blockDim.x) ln_sm[h] = 0.0f;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarp = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long r = warp; r < R; r += nwarp) {
        const float* xr = x + r * H;
        const float mean = stats[2 * r], rstd = stats[2 * r + 1];
        const long long bb = Tt > 0 ? r / Tt : 0;
        const int t = Tt > 0 ? (int)(r - bb * Tt) : 0;
        float m1 = 0.0f, m2 = 0.0f;
        for (int h = lane; h < H; h += 32) {
            const float d = Tt > 0 ? dy[(bb * H + h) * Tt + t] : dy[r * H + h];
            const float xh = (xr[h] - mean) * rstd, dg_ = d * g[h];
            m1 += dg_;
            m2 = fmaf(dg_, xh, m2);
            atomicAdd(dgs + h, d * xh);
            atomicAdd(dbs + h, d);
        }
        m1 = warp_sum(m1) / (float)H;
        m2 = warp_sum(m2) / (float)H;
        for (int h = lane; h < H; h += 32) {
            const float d = Tt > 0 ? dy[(bb * H + h) * Tt + t] : dy[r * H + h];
            const float xh = (xr[h] - mean) * rstd, dg_ = d * g[h];
            const float base = res ? res[r * H + h] : 0.0f;
            dx[r * H + h] = fmaf(rstd, dg_ - m1 - xh * m2, base);
        }
    }
    __syncthreads();
    for (int h = threadIdx.x; h < H; h += blockDim.x) { atomicAdd(dg + h, dgs[h]); atomicAdd(db + h, dbs[h]); }
}

// ------------------------------------------------------------------------------------------ BatchNorm1d over [N, C, L]
// sums[c] += sum_{n,l} a,  sums[C + c] += sum a^2,   a = act(u)          (one warp per (n, c) row of L elements)
template <int ACT>
__global__ void __launch_bounds__(kT) bn_stats_kernel(const float* __restrict__ u, double* sums, long long NC, int C, int L) {
    extern __shared__ double bn_sm[];
    for (int c = threadIdx.x; c < 2 * C; c += blockDim.x) bn_sm[c] = 0.0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarp = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long row = warp; row < NC; row += nwarp) {
        const int c = (int)(row % C);
        const float* ur = u + row * L;
        float s = 0.0f, q = 0.0f;
        for (int l = lane; l < L; l += 32) { const float a = actf<ACT>(ur[l]); s += a; q = fmaf(a, a, q); }
        s = warp_sum(s); q = warp_sum(q);
        if (lane == 0) { atomicAdd(bn_sm + c, (double)s); atomicAdd(bn_sm + C + c, (double)q); }
    }
    __syncthreads();
    for (int c = threadIdx.x; c < 2 * C; c += blockDim.x)
        if (bn_sm[c] != 0.0) atomicAdd(sums + c, bn_sm[c]);
}

// y = act(u) * scale[c] + shift[c]
template <int ACT>
__global__ void __launch_bounds__(kT) bn_apply_kernel(const float* __restrict__ u, const float* __restrict__ bn, float* __restrict__ y,
                                                      long long total, int C, int L) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int c = (int)((i / L) % C);
        y[i] = fmaf(actf<ACT>(u[i]), bn[c], bn[C + c]);
    }
}

// sums[c] += sum dR,  sums[C + c] += sum dR * xhat,   xhat = act(u) * xs[c] + xo[c]
template <int ACT>
__global__ void __launch_bounds__(kT) bn_bwd_reduce_kernel(const float* __restrict__ u, const float* __restrict__ bn, const float* __restrict__ dy,
                                                           double* sums, long long NC, int C, int L) {
    extern __shared__ double bn_sm[];
    for (int c = threadIdx.x; c < 2 * C; c += blockDim.x) bn_sm[c] = 0.0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarp = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long row = warp; row < NC; row += nwarp) {
        const int c = (int)(row % C);
        const float xs = bn[2 * C + c], xo = bn[3 * C + c];
        float s = 0.0f, q = 0.0f;
        for (int l = lane; l < L; l += 32) {
            const float d = dy[row * L + l];
            s += d;
            q = fmaf(d, fmaf(actf<ACT>(u[row * L + l]), xs, xo), q);
        }
        s = warp_sum(s); q = warp_sum(q);
        if (lane == 0) { atomicAdd(bn_sm + c, (double)s); atomicAdd(bn_sm + C + c, (double)q); }
    }
    __syncthreads();
    for (int c = threadIdx.x; c < 2 * C; c += blockDim.x)
        if (bn_sm[c] != 0.0) atomicAdd(sums + c, bn_sm[c]);
}

// du = k1[c] * (dR - k2[c] - xhat * k3[c]) * act'(u)        (du may alias dy)
template <int ACT>
__global__ void __launch_bounds__(kT) bn_bwd_apply_kernel(const float* __restrict__ u, const float* __restrict__ bn, const float* __restrict__ coef,
                                                          const float* dy, float* du, long long total, int C, int L) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int c = (int)((i / L) % C);
        float a;
        const float da = actf_grad<ACT>(u[i], &a);
        const float xh = fmaf(a, bn[2 * C + c], bn[3 * C + c]);
        du[i] = coef[c] * (dy[i] - coef[C + c] - xh * coef[2 * C + c]) * da;
    }
}

// ------------------------------------------------------------------------------------------ BN affine -> SE -> residual
struct SeResArgs {
    const float *x, *v, *bn, *se1, *se2, *dout;
    float *out, *dv, *g_se1, *g_se2;
    int B, T, H, rr, use_max, trans, by_h;
};

// shared: y tile [T*H] | s [T] | gate [T] | dq [T] | ds [T] | z [rr] | dz [rr] | am [T] (int) | gs1 [rr*T] | gs2 [T*rr]
__device__ __forceinline__ void se_tile_forward(const SeResArgs& a, int b, float* ys, float* s, float* gate, float* z, int* am) {
    const int T = a.T, H = a.H, rr = a.rr, Cn = a.by_h ? H : T;
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
    for (int i = tid; i < T * H; i += nt) {
        const int t = i / H, h = i - t * H;
        const float vv = a.trans ? a.v[((size_t)b * H + h) * T + t] : a.v[((size_t)b * T + t) * H + h];
        const int c = a.by_h ? h : t;
        ys[i] = fmaf(vv, a.bn[c], a.bn[Cn + c]);
    }
    __syncthreads();
    for (int t = warp; t < T; t += nw) {
        if (a.use_max) {
            float m = -INFINITY;
            int mi = 0x7fffffff;
            for (int h = lane; h < H; h += 32) { const float v = ys[t * H + h]; if (v > m) { m = v; mi = h; } }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float om = __shfl_xor_sync(0xffffffffu, m, o);
                const int oi = __shfl_xor_sync(0xffffffffu, mi, o);
                if (om > m || (om == m && oi < mi)) { m = om; mi = oi; }
            }
            if (lane == 0) { s[t] = m; am[t] = mi; }
        } else {
            float v = 0.0f;
            for (int h = lane; h < H; h += 32) v += ys[t * H + h];
            v = warp_sum(v);
            if (lane == 0) s[t] = v / (float)H;
        }
    }
    __syncthreads();
    if (rr > 0) {
        if (tid < rr) {
            float acc = 0.0f;
            for (int t = 0; t < T; ++t) acc = fmaf(a.se1[tid * T + t], s[t], acc);
            z[tid] = acc;
        }
        __syncthreads();
        if (tid < T) {
            float q = 0.0f;
            for (int k = 0; k < rr; ++k) q = fmaf(a.se2[tid * rr + k], fmaxf(z[k], 0.0f), q);
            gate[tid] = sigmoidf_(q);
        }
    } else if (tid < T) {
        gate[tid] = 1.0f;
    }
    __syncthreads();
}

// out = x + SE(v * scale + shift)       (mlp_mixer.py:152-155 resp. :161-164 with reg2 = BatchNorm1d folded in)
__global__ void __launch_bounds__(kT) se_res_fwd_kernel(const SeResArgs a) {
    extern __shared__ float se_sm[];
    const int T = a.T, H = a.H, rr = a.rr;
    float* ys = se_sm;
    float* s = ys + T * H;
    float* gate = s + T;
    float* z = gate + 3 * T;
    int* am = reinterpret_cast<int*>(z + 2 * (rr > 0 ? rr : 1));
    for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
        se_tile_forward(a, b, ys, s, gate, z, am);
        for (int i = threadIdx.x; i < T * H; i += blockDim.x) {
            const size_t gi = (size_t)b * T * H + i;
            a.out[gi] = fmaf(ys[i], gate[i / H], a.x[gi]);
        }
        __syncthreads();
    }
}

// dv (in v's layout) = d(out)/d(v * scale + shift) applied to dout: SE backward; SE weight gradients accumulated
__global__ void __launch_bounds__(kT) se_res_bwd_kernel(const SeResArgs a) {
    extern __shared__ float se_sm[];
    const int T = a.T, H = a.H, rr = a.rr, rr1 = rr > 0 ? rr : 1;
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
    float* ys = se_sm;
    float* s = ys + T * H;
    float* gate = s + T;
    float* dq = gate + T;
    float* ds = dq + T;
    float* z = ds + T;
    float* dz = z + rr1;
    int* am = reinterpret_cast<int*>(dz + rr1);
    float* gs1 = reinterpret_cast<float*>(am + T);
    float* gs2 = gs1 + rr1 * T;
    for (int i = tid; i < 2 * rr1 * T; i += nt) gs1[i] = 0.0f;
    __syncthreads();
    for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
        se_tile_forward(a, b, ys, s, gate, z, am);
        const float* dob = a.dout + (size_t)b * T * H;
        if (rr > 0) {
            for (int t = warp; t < T; t += nw) {
                float v = 0.0f;
                for (int h = lane; h < H; h += 32) v = fmaf(dob[t * H + h], ys[t * H + h], v);
                v = warp_sum(v);
                if (lane == 0) dq[t] = v * gate[t] * (1.0f - gate[t]);
            }
            __syncthreads();
            if (tid < rr) {
                float da = 0.0f;
                for (int t = 0; t < T; ++t) da = fmaf(dq[t], a.se2[t * rr + tid], da);
                dz[tid] = z[tid] > 0.0f ? da : 0.0f;
            }
            __syncthreads();
            if (tid < T) {
                float acc = 0.0f;
                for (int k = 0; k < rr; ++k) acc = fmaf(dz[k], a.se1[k * T + tid], acc);
                ds[tid] = acc;
            }
            for (int i = tid; i < rr * T; i += nt) {
                const int k = i / T, t = i - k * T;
                gs1[i] = fmaf(dz[k], s[t], gs1[i]);                          // dS1[k][t]
                gs2[t * rr + k] = fmaf(dq[t], fmaxf(z[k], 0.0f), gs2[t * rr + k]);   // dS2[t][k]
            }
            __syncthreads();
        }
        for (int i = tid; i < T * H; i += nt) {
            const int t = i / H, h = i - t * H;
            float d = dob[i] * gate[t];
            if (rr > 0) d += a.use_max ? (h == am[t] ? ds[t] : 0.0f) : ds[t] / (float)H;
            if (a.trans) a.dv[((size_t)b * H + h) * T + t] = d; else a.dv[((size_t)b * T + t) * H + h] = d;
        }
        __syncthreads();
    }
    if (rr > 0)
        for (int i = tid; i < rr * T; i += nt) { atomicAdd(a.g_se1 + i, gs1[i]); atomicAdd(a.g_se2 + i, gs2[i]); }
}

int act_code(int act) {    // MMX_ACT_GELU / MMX_ACT_MISH / negative: identity
    return act < 0 ? ACT_ID : (act == MMX_ACT_GELU ? ACT_GELU : (act == MMX_ACT_MISH ? ACT_MISH : -1));
}
size_t se_smem(int T, int H, int rr) {
    const int rr1 = rr > 0 ? rr : 1;
    return (size_t)(T * H + 5 * T + 2 * rr1 + 2 * rr1 * T + 8) * 4;
}
int check_se(int B, int T, int H, int rr, size_t* smem, const char* what) {
    if (B <= 0 || T <= 0 || H <= 0 || rr < 0) return fail(MMX_E_INVALID, "%s: bad sizes", what);
    if (T > kT || rr > kT) return fail(MMX_E_UNSUPPORTED, "%s: seq_len %d / SE width %d above %d", what, T, rr, kT);
    *smem = se_smem(T, H, rr);
    if (*smem > (size_t)dev_info().max_smem) return fail(MMX_E_UNSUPPORTED, "%s: a [%d x %d] tile does not fit shared memory", what, T, H);
    return MMX_OK;
}
}  // namespace

extern "C" int mmx_ln_fwd(long long rows, int H, int Tt, const float* x, const float* g, const float* b, float* y, float* stats, void* stream) {
    if (!x || !g || !b || !y || !stats) return fail(MMX_E_INVALID, "mmx_ln_fwd: null tensor");
    if (rows <= 0 || H <= 0 || Tt < 0 || (Tt > 0 && rows % Tt)) return fail(MMX_E_INVALID, "mmx_ln_fwd: bad sizes");
    return launch_kernel(ln_fwd_kernel, capped_grid(dev_info(), rows, kT / 32, 8), kT, 0, stream, kNoPdl, x, g, b, y, stats, rows, H, Tt);
}

extern "C" int mmx_ln_bwd(long long rows, int H, int Tt, const float* x, const float* stats, const float* g, const float* dy, const float* res,
                          float* dx, float* dg, float* db, void* stream) {
    if (!x || !stats || !g || !dy || !dx || !dg || !db) return fail(MMX_E_INVALID, "mmx_ln_bwd: null tensor");
    if (rows <= 0 || H <= 0 || Tt < 0 || (Tt > 0 && rows % Tt)) return fail(MMX_E_INVALID, "mmx_ln_bwd: bad sizes");
    if ((size_t)H * 8 > 48 * 1024) return fail(MMX_E_UNSUPPORTED, "mmx_ln_bwd: H = %d too wide", H);
    const int grid = capped_grid(dev_info(), rows, 64, 4);      // >= 8 rows per warp: the per-CTA flush of dg / db is amortised
    return launch_kernel(ln_bwd_kernel, grid, kT, (size_t)H * 8, stream, kNoPdl, x, stats, g, dy, res, dx, dg, db, rows, H, Tt);
}

#define MMX_BN_KERNEL(kern) (code == ACT_GELU ? kern<ACT_GELU> : code == ACT_MISH ? kern<ACT_MISH> : kern<ACT_ID>)

static int check_bn(long long N, int C, int L, int act, const char* what) {
    if (N <= 0 || C <= 0 || L <= 0) return fail(MMX_E_INVALID, "%s: bad sizes", what);
    if (act_code(act) < 0) return fail(MMX_E_INVALID, "Unknown activation function type: %d", act);
    if (C > 2048) return fail(MMX_E_UNSUPPORTED, "%s: %d channels", what, C);
    return MMX_OK;
}

extern "C" int mmx_bn1d_stats(long long N, int C, int L, int act, const float* u, double* sums, void* stream) {
    if (!u || !sums) return fail(MMX_E_INVALID, "mmx_bn1d_stats: null tensor");
    int rc = check_bn(N, C, L, act, "mmx_bn1d_stats");
    if (rc) return rc;
    const int code = act_code(act);
    const long long NC = N * C;
    return launch_kernel(MMX_BN_KERNEL(bn_stats_kernel), capped_grid(dev_info(), NC, 128, 4), kT, (size_t)C * 16, stream, kNoPdl, u, sums, NC, C, L);
}

extern "C" int mmx_bn1d_apply(long long N, int C, int L, int act, const float* u, const float* bn, float* y, void* stream) {
    if (!u || !bn || !y) return fail(MMX_E_INVALID, "mmx_bn1d_apply: null tensor");
    int rc = check_bn(N, C, L, act, "mmx_bn1d_apply");
    if (rc) return rc;
    const int code = act_code(act);
    const long long total = N * C * L;
    return launch_kernel(MMX_BN_KERNEL(bn_apply_kernel), capped_grid(dev_info(), total, kT * 4, 8), kT, 0, stream, kNoPdl, u, bn, y, total, C, L);
}

extern "C" int mmx_bn1d_bwd_reduce(long long N, int C, int L, int act, const float* u, const float* bn, const float* dy, double* sums, void* stream) {
    if (!u || !bn || !dy || !sums) return fail(MMX_E_INVALID, "mmx_bn1d_bwd_reduce: null tensor");
    int rc = check_bn(N, C, L, act, "mmx_bn1d_bwd_reduce");
    if (rc) return rc;
    const int code = act_code(act);
    const long long NC = N * C;
    return launch_kernel(MMX_BN_KERNEL(bn_bwd_reduce_kernel), capped_grid(dev_info(), NC, 128, 4), kT, (size_t)C * 16, stream, kNoPdl, u, bn, dy, sums,
                         NC, C, L);
}

extern "C" int mmx_bn1d_bwd_apply(long long N, int C, int L, int act, const float* u, const float* bn, const float* coef, const float* dy,
                                  float* du, void* stream) {
    if (!u || !bn || !coef || !dy || !du) return fail(MMX_E_INVALID, "mmx_bn1d_bwd_apply: null tensor");
    int rc = check_bn(N, C, L, act, "mmx_bn1d_bwd_apply");
    if (rc) return rc;
    const int code = act_code(act);
    const long long total = N * C * L;
    return launch_kernel(MMX_BN_KERNEL(bn_bwd_apply_kernel), capped_grid(dev_info(), total, kT * 4, 8), kT, 0, stream, kNoPdl, u, bn, coef, dy, du,
                         total, C, L);
}

extern "C" int mmx_se_res_fwd(int B, int T, int H, int se_hidden, int use_max_pooling, int v_transposed, int affine_by_h, const float* x,
                              const float* v, const float* bn, const float* se_w1, const float* se_w2, float* out, void* stream) {
    if (!x || !v || !bn || !out || (se_hidden > 0 && (!se_w1 || !se_w2))) return fail(MMX_E_INVALID, "mmx_se_res_fwd: null tensor");
    size_t smem;
    int rc = check_se(B, T, H, se_hidden, &smem, "mmx_se_res_fwd");
    if (rc) return rc;
    SeResArgs a = {};
    a.x = x; a.v = v; a.bn = bn; a.se1 = se_w1; a.se2 = se_w2; a.out = out;
    a.B = B; a.T = T; a.H = H; a.rr = se_hidden; a.use_max = use_max_pooling; a.trans = v_transposed; a.by_h = affine_by_h;
    return launch_kernel(se_res_fwd_kernel, capped_grid(dev_info(), B, 1, 8), kT, smem, stream, kNoPdl, a);
}

extern "C" int mmx_se_res_bwd(int B, int T, int H, int se_hidden, int use_max_pooling, int v_transposed, int affine_by_h, const float* v,
                              const float* bn, const float* se_w1, const float* se_w2, const float* dout, float* g_se_w1, float* g_se_w2,
                              float* dv, void* stream) {
    if (!v || !bn || !dout || !dv || (se_hidden > 0 && (!se_w1 || !se_w2 || !g_se_w1 || !g_se_w2))) return fail(MMX_E_INVALID, "mmx_se_res_bwd: null tensor");
    size_t smem;
    int rc = check_se(B, T, H, se_hidden, &smem, "mmx_se_res_bwd");
    if (rc) return rc;
    SeResArgs a = {};
    a.v = v; a.bn = bn; a.se1 = se_w1; a.se2 = se_w2; a.dout = dout; a.dv = dv; a.g_se1 = g_se_w1; a.g_se2 = g_se_w2;
    a.B = B; a.T = T; a.H = H; a.rr = se_hidden; a.use_max = use_max_pooling; a.trans = v_transposed; a.by_h = affine_by_h;
    return launch_kernel(se_res_bwd_kernel, capped_grid(dev_info(), B, 1, 4), kT, smem, stream, kNoPdl, a);     // B >= 1: check_se
}
#endif
