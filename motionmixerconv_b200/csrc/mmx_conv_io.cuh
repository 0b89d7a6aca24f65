// ConvMixer input / output stages: PoseEncoder (optional harmonic embedding), the model head and
// the "once"-mode squeeze-excitation tail.
//
// Reference arithmetic: conv_mixer/encoding/positional_encoder.py:79-97 (PoseEncoder.forward),
// h36m/conv_mixer_model.py:455-463 (LN -> conv_out -> project_channels -> GELU -> fc_out) and
// :287-292 with mode_conv="once" (y = x + se(x)); restated in oracle/mixer_np.py.
#pragma once
#include "mmx_conv.cuh"

namespace mmx {

#if defined(MMX_HOST_EMU)
MMX_D float mul_rn(float a, float b) { volatile float p = a * b; return p; }
#else
MMX_D float mul_rn(float a, float b) { return __fmul_rn(a, b); }   // ONE fp32 multiply, never contracted
#endif


// ------------------------------------------------------------------------------------------
// Harmonic phases by exact angle doubling.
// frequencies[h] = omega0 * 2^h (positional_encoder.py:54-57), so the fp32 argument of harmonic h is
// a_h = fl32(x*f_h) = fl32(x*f_0) * 2^h EXACTLY (scaling by a power of two commutes with rounding).  Instead of one
// Payne-Hanek reduction per (x, h) -- arguments reach 1e17 -- the phase frac(a_0 / 2pi) is formed ONCE as a 128-bit
// fixed-point fraction (24-bit mantissa x 128 bits of 1/2pi) and harmonic h is a left shift by h bits.  sin/cos are then
// evaluated on a float-float reduced argument in [-pi, pi) (fast path of sincosf), matching sinf(a_h)/cosf(a_h) of the
// exact fp32 argument to ~2 ulp.  Used only when the frequency table really is f_0 * 2^h (checked on the device).
// ------------------------------------------------------------------------------------------
struct Phase128 { uint32_t w0, w1, w2, w3; };   // w0 most significant

#if defined(MMX_HOST_EMU)
static const uint32_t kInv2PiBits[13] =
#else
static __device__ __constant__ uint32_t kInv2PiBits[13] =
#endif
    {0u, 0u, 0u, 0u, 0x28be60dbu, 0x9391054au, 0x7f09d5f4u, 0x7d4d3770u, 0x36d8a566u, 0x4f10e410u, 0x7f9458eau, 0xf7aef158u, 0x6dc91b8eu};

MMX_D uint32_t f2u(float f) {
#if defined(MMX_HOST_EMU)
    uint32_t u; memcpy(&u, &f, 4); return u;
#else
    return __float_as_uint(f);
#endif
}

// phase of |a|; returns false when a is zero / denormal / tiny / non-finite (caller evaluates sinf / cosf directly)
MMX_D bool phase_init(float a, Phase128* ph, bool* neg) {
    const uint32_t bits = f2u(a);
    const int ex = (int)((bits >> 23) & 0xffu);
    *neg = (bits >> 31) != 0u;
    if (ex < 22 || ex == 255) return false;
    const uint32_t m = (bits & 0x7fffffu) | 0x800000u;   // |a| = m * 2^(ex-150)
    const int sh = ex - 22;                              // bits of (1/2pi * 2^-128) shifted out as integer part: 128 + (ex-150)
    const int wo = sh >> 5, bo = sh & 31;
    uint32_t k[4];
    MMX_UNROLL
    for (int i = 0; i < 4; ++i) {
        const uint32_t hi = kInv2PiBits[wo + i], lo = kInv2PiBits[wo + i + 1];
        k[i] = bo ? (hi << bo) | (lo >> (32 - bo)) : hi;
    }
    uint64_t t = (uint64_t)m * k[3];
    ph->w3 = (uint32_t)t; t = (uint64_t)m * k[2] + (t >> 32);
    ph->w2 = (uint32_t)t; t = (uint64_t)m * k[1] + (t >> 32);
    ph->w1 = (uint32_t)t; t = (uint64_t)m * k[0] + (t >> 32);
    ph->w0 = (uint32_t)t;
    return true;
}
MMX_D void phase_shl(Phase128* p, int n) {   // multiply the angle by 2^n (0 <= n < 128)
    uint32_t w[8] = {p->w0, p->w1, p->w2, p->w3, 0u, 0u, 0u, 0u};
    const int wo = n >> 5, bo = n & 31;
    uint32_t r[4];
    MMX_UNROLL
    for (int i = 0; i < 4; ++i) {
        uint32_t hi = 0u, lo = 0u;
        MMX_UNROLL
        for (int j = 0; j < 4; ++j) { if (wo == j) { hi = w[i + j]; lo = w[i + j + 1]; } }
        r[i] = bo ? (hi << bo) | (lo >> (32 - bo)) : hi;
    }
    p->w0 = r[0]; p->w1 = r[1]; p->w2 = r[2]; p->w3 = r[3];
}
MMX_D void phase_double(Phase128* p) {
    p->w0 = (p->w0 << 1) | (p->w1 >> 31); p->w1 = (p->w1 << 1) | (p->w2 >> 31);
    p->w2 = (p->w2 << 1) | (p->w3 >> 31); p->w3 <<= 1;
}
MMX_D void phase_sincos(const Phase128& p, bool neg, float* s, float* c) {
    const float phi_hi = (float)(int32_t)(p.w0 & 0xffffff00u) * 2.3283064365386963e-10f;              // * 2^-32, exact
    const float phi_lo = (float)(((p.w0 & 0xffu) << 16) | (p.w1 >> 16)) * 1.3877787807814457e-17f;    // * 2^-56, exact
    const float C_HI = 6.2831854820251465f, C_LO = -1.7484556000744883e-07f;                          // 2pi = C_HI + C_LO
    const float r_hi = phi_hi * C_HI;
    const float r_lo = fmaf(phi_hi, C_HI, -r_hi) + fmaf(phi_hi, C_LO, phi_lo * C_HI);
    const float s0 = sinf(r_hi), c0 = cosf(r_hi);
    const float sv = fmaf(r_lo, c0, s0);
    *s = neg ? -sv : sv;
    *c = fmaf(-r_lo, s0, c0);
}

// sin / cos of fl32(x * freq[h]) for h = h0 .. h0+n-1 of one input value; out_s / out_c are strided by 1
MMX_D void harmonics(float x, const float* freq, bool pow2, int h0, int n, float* out_s, float* out_c) {
    Phase128 ph;
    bool neg;
    if (pow2 && phase_init(mul_rn(x, freq[0]), &ph, &neg)) {
        phase_shl(&ph, h0);
        for (int i = 0; i < n; ++i) {
            phase_sincos(ph, neg, out_s + i, out_c + i);
            phase_double(&ph);
        }
    } else {
        for (int i = 0; i < n; ++i) {
            const float arg = mul_rn(x, freq[h0 + i]);
            out_s[i] = sinf(arg); out_c[i] = cosf(arg);
        }
    }
}

// 1 when freq[h] == freq[0] * 2^h for every h < Hn <= 64 (exact), else 0
MMX_D int freq_is_pow2_ladder(const float* freq, int Hn) {
    if (Hn > 64 || !(freq[0] > 0.0f)) return 0;
    for (int h = 1; h < Hn; ++h)
        if (freq[h] != ldexpf(freq[0], h)) return 0;
    return 1;
}

// ==========================================================================================
// "once"-mode tail:  y = x + SE(x)   (or 2x without SE)        conv_mixer_model.py:287-292
// ==========================================================================================
struct SeTailDims { int B, C, T, E, rr, S, use_se, use_max; };
struct SeTailSmem { int se1, se2, part, part2, pool, gate, amax, z, dq, dz, ds, a_se1, a_se2, total; };
MMX_HD SeTailSmem se_tail_smem(const SeTailDims& d) {
    SeTailSmem L;
    const int rr = imax(d.rr, 1), ST = d.S * d.T;
    int o = 0;
    auto take = [&](int n) { int r = o; o += round_up(n, 4); return r; };
    L.se1 = take(rr * d.T); L.se2 = take(d.T * rr);
    L.part = take(ST * kParts); L.part2 = take(ST * kParts);
    L.pool = take(ST); L.gate = take(ST); L.amax = take(ST); L.z = take(d.S * rr);
    L.dq = take(ST); L.dz = take(d.S * rr); L.ds = take(ST);
    L.a_se1 = take(rr * d.T); L.a_se2 = take(d.T * rr);
    L.total = o;
    return L;
}
struct SeTailArgs {
    SeTailDims d;
    const float *se1, *se2;   // parameters (null without SE)
    float *g_se1, *g_se2;     // gradient accumulators (backward)
    const float* x;
    const float* dy;          // backward only
    float* out;               // forward: y, backward: dx
};

MMX_D void se_tail_fwd_body(Exec& ex, const SeTailArgs& a) {
    const SeTailDims& d = a.d;
    const SeTailSmem L = se_tail_smem(d);
    float* sm = ex.smem;
    const int nthr = ex.nthr, C = d.C, T = d.T, E = d.E, S = d.S, rr = d.rr;
    if (d.use_se)
        ex.phase([&](int tid) { copy_vec(tid, nthr, sm + L.se1, a.se1, rr * T); copy_vec(tid, nthr, sm + L.se2, a.se2, T * rr); });
    const int ntiles = (d.B + S - 1) / S;
    for (int tile = ex.bid; tile < ntiles; tile += ex.nblk) {
        const long long seq0 = (long long)tile * S;
        const int ns = imin(S, d.B - (int)seq0), nr = ns * C * T;
        const float* xg = a.x + (size_t)seq0 * C * T * E;
        float* yg = a.out + (size_t)seq0 * C * T * E;
        if (d.use_se) {
            ex.phase([&](int tid) {
                for (int i = tid; i < ns * T * kParts; i += nthr) {
                    const int st = i / kParts, p = i - st * kParts, s = st / T, t = st - s * T;
                    se_pool_part(xg + ((size_t)(s * C) * T + t) * E, T * E, C, E, p, d.use_max, sm + L.part + i, sm + L.part2 + i);
                }
            });
            ex.phase([&](int tid) {
                for (int st = tid; st < ns * T; st += nthr)
                    se_pool_combine(sm + L.part + st * kParts, sm + L.part2 + st * kParts, C * E, d.use_max, sm + L.pool + st, sm + L.amax + st);
            });
            ex.phase([&](int tid) {
                for (int st = tid; st < ns * T; st += nthr) {
                    const int s = st / T, t = st - s * T;
                    sm[L.gate + st] = se_excite(sm + L.se1, sm + L.se2, sm + L.pool + s * T, T, rr, t, nullptr);
                }
            });
        }
        ex.phase([&](int tid) {
            for (int i = tid; i < nr * E; i += nthr) {
                const int r = i / E, sc = r / T, t = r - sc * T, s = sc / C;
                const float g = d.use_se ? sm[L.gate + s * T + t] : 1.0f;
                const float v = xg[i];
                yg[i] = fmaf(g, v, v);
            }
        });
    }
}

MMX_D void se_tail_bwd_body(Exec& ex, const SeTailArgs& a) {
    const SeTailDims& d = a.d;
    const SeTailSmem L = se_tail_smem(d);
    float* sm = ex.smem;
    const int nthr = ex.nthr, C = d.C, T = d.T, E = d.E, S = d.S, rr = d.rr;
    const float invCE = 1.0f / (float)(C * E);
    if (d.use_se)
        ex.phase([&](int tid) {
            copy_vec(tid, nthr, sm + L.se1, a.se1, rr * T); copy_vec(tid, nthr, sm + L.se2, a.se2, T * rr);
            zero_vec(tid, nthr, sm + L.a_se1, rr * T); zero_vec(tid, nthr, sm + L.a_se2, T * rr);
        });
    const int ntiles = (d.B + S - 1) / S;
    for (int tile = ex.bid; tile < ntiles; tile += ex.nblk) {
        const long long seq0 = (long long)tile * S;
        const int ns = imin(S, d.B - (int)seq0), nr = ns * C * T;
        const float* xg = a.x + (size_t)seq0 * C * T * E;
        const float* dyg = a.dy + (size_t)seq0 * C * T * E;
        float* dxg = a.out + (size_t)seq0 * C * T * E;
        if (d.use_se) {
            ex.phase([&](int tid) {
                for (int i = tid; i < ns * T * kParts; i += nthr) {
                    const int st = i / kParts, p = i - st * kParts, s = st / T, t = st - s * T;
                    se_pool_part(xg + ((size_t)(s * C) * T + t) * E, T * E, C, E, p, d.use_max, sm + L.part + i, sm + L.part2 + i);
                }
            });
            ex.phase([&](int tid) {
                for (int st = tid; st < ns * T; st += nthr)
                    se_pool_combine(sm + L.part + st * kParts, sm + L.part2 + st * kParts, C * E, d.use_max, sm + L.pool + st, sm + L.amax + st);
            });
            ex.phase([&](int tid) {   // dgate partials: sum_{c,e} dy * x
                for (int i = tid; i < ns * T * kParts; i += nthr) {
                    const int st = i / kParts, p = i - st * kParts, s = st / T, t = st - s * T;
                    float dg = 0.0f;
                    for (int c = 0; c < C; ++c) {
                        const size_t off = ((size_t)(s * C + c) * T + t) * E;
                        for (int h = 4 * p; h < E; h += 4 * kParts) {
                            const int n = imin(4, E - h);
                            for (int k = 0; k < n; ++k) dg = fmaf(dyg[off + h + k], xg[off + h + k], dg);
                        }
                    }
                    sm[L.part + i] = dg;
                }
                for (int st = tid; st < ns * T; st += nthr) {
                    const int s = st / T, t = st - s * T;
                    sm[L.gate + st] = se_excite(sm + L.se1, sm + L.se2, sm + L.pool + s * T, T, rr, t, sm + L.z + s * rr);
                }
            });
            ex.phase([&](int tid) {
                for (int st = tid; st < ns * T; st += nthr) sm[L.dq + st] = sum_parts(sm + L.part + st * kParts);
            });
            se_bwd_phases(ex, sm, T, rr, ns, L.se1, L.se2, L.dq, L.dz, L.gate, L.pool, L.z, L.ds, L.a_se1, L.a_se2);
        }
        ex.phase([&](int tid) {
            for (int i = tid; i < nr * E; i += nthr) {
                const int r = i / E, e = i - r * E, sc = r / T, t = r - sc * T, s = sc / C, c = sc - s * C;
                const float g = d.use_se ? sm[L.gate + s * T + t] : 1.0f;
                const float dv = dyg[i];
                float v = fmaf(g, dv, dv);
                if (d.use_se) {
                    if (d.use_max) { if (c * E + e == (int)sm[L.amax + s * T + t]) v += sm[L.ds + s * T + t]; }
                    else v = fmaf(sm[L.ds + s * T + t], invCE, v);
                }
                dxg[i] = v;
            }
        });
    }
    if (d.use_se)
        ex.phase([&](int tid) {
            for (int i = tid; i < T * rr; i += nthr) { red_add(a.g_se1 + i, sm[L.a_se1 + i]); red_add(a.g_se2 + i, sm[L.a_se2 + i]); }
        });
}

// ==========================================================================================
// PoseEncoder                                             positional_encoder.py:79-97
//   emb[r][d*Hn+h] = sin(x[r][d]*f[h]),  emb[r][Hn*D + d*Hn+h] = cos(..)     (Hn > 0; else emb = x)
//   m[r][:] = W emb[r][:] + b ;  y[b][c][t][:] = m[b*T+t][:] * wc[c] + bc[c]
// ==========================================================================================
struct EncDims {
    int B, T, D, E, C, Hn;
    int K;        // embedding width: Hn > 0 ? 2*Hn*D : D
    int KC;       // embedding columns per chunk (multiple of 4)
    int DC;       // harmonic embedding: input dimensions per chunk (a chunk = their sin AND cos columns, KC >= 2*DC*HC)
    int HC;       // harmonic embedding: harmonics per chunk; HC < Hn (then DC = 1) splits one input dimension over several chunks
    int R;        // frames (rows of x) per CTA tile
};
struct EncW { float *freq, *w, *b, *wc, *bc; };   // frequencies[Hn], embed_mlp.{weight[E,K],bias[E]}, channelUpscaling.{weight[C,1],bias[C]}
struct EncSmem { int PKC, PE, PD, x, emb, w, m, b, wc, bc, freq, flag, total; };
MMX_HD EncSmem enc_smem(const EncDims& d) {
    EncSmem L;
    L.PKC = pitch_of(d.KC); L.PE = pitch_of(d.E); L.PD = round_up(d.D, 4);
    int o = 0;
    auto take = [&](int n) { int r = o; o += round_up(n, 4); return r; };
    L.x = take(d.R * L.PD); L.emb = take(d.R * L.PKC); L.w = take(d.E * L.PKC); L.m = take(d.R * L.PE);
    L.b = take(d.E); L.wc = take(8); L.bc = take(8); L.freq = take(imax(d.Hn, 1)); L.flag = take(4);
    L.total = o;
    return L;
}

// embedding value of global column kk for the frame whose inputs are xr[0..D)
MMX_D float enc_embed(const float* xr, const float* freq, int D, int Hn, int kk) {
    if (Hn <= 0) return xr[kk];
    const int half = Hn * D;
    const int k2 = kk < half ? kk : kk - half;
    const int dd = k2 / Hn, h = k2 - dd * Hn;
    const float arg = mul_rn(xr[dd], freq[h]);
    return kk < half ? sinf(arg) : cosf(arg);
}

struct EncFwdArgs { EncDims d; EncW w; const float* x; float* m; float* y; };   // m: [B*T,E] saved for the backward

struct EncFwdRegs { float acc[4][4]; };

MMX_D void enc_fwd_body(Exec& ex, const EncFwdArgs& a) {
    const EncDims& d = a.d;
    const EncSmem L = enc_smem(d);
    float* sm = ex.smem;
    const int nthr = ex.nthr, D = d.D, E = d.E, C = d.C, T = d.T, K = d.K, KC = d.KC, R = d.R, PKC = L.PKC, PE = L.PE;
    const int rows = d.B * T;
    const int Hn = d.Hn, DC = d.DC, HC = d.HC;
    const int nseg = Hn > 0 ? (Hn + HC - 1) / HC : 1;     // harmonic segments per group of DC input dimensions
    const int nchunks = Hn > 0 ? ((D + DC - 1) / DC) * nseg : (K + KC - 1) / KC;
    PerThread<EncFwdRegs> regs(ex);
    ex.phase([&](int tid) {
        copy_vec(tid, nthr, sm + L.b, a.w.b, E);
        for (int i = tid; i < 8; i += nthr) { sm[L.wc + i] = i < C ? a.w.wc[i] : 0.0f; sm[L.bc + i] = i < C ? a.w.bc[i] : 0.0f; }
        if (Hn > 0) copy_vec(tid, nthr, sm + L.freq, a.w.freq, Hn);
        if (tid == 0) sm[L.flag] = Hn > 0 ? (float)freq_is_pow2_ladder(a.w.freq, Hn) : 0.0f;
    });
    const int ntiles = (rows + R - 1) / R;
    for (int tile = ex.bid; tile < ntiles; tile += ex.nblk) {
        const int row0 = tile * R, nr = imin(R, rows - row0);
        // output tiling of m[nr][E]: 4x4 thread tiles with strided ownership, K of a chunk split over `ks` thread groups
        const int n_rt = (nr + 3) >> 2, n_ct = (E + 3) >> 2, tiles = n_rt * n_ct;
        const int ksplit = imax(1, imin(8, nthr / tiles));
        ex.phase([&](int tid) {
            for (int i = tid; i < nr * L.PD; i += nthr) {
                const int r = i / L.PD, c = i - r * L.PD;
                sm[L.x + i] = c < D ? a.x[(size_t)(row0 + r) * D + c] : 0.0f;
            }
            zero_vec(tid, nthr, sm + L.m, nr * PE);
            EncFwdRegs& rg = regs[tid];
            MMX_UNROLL
            for (int i = 0; i < 4; ++i)
                MMX_UNROLL
                for (int j = 0; j < 4; ++j) rg.acc[i][j] = 0.0f;
        });
        for (int ch = 0; ch < nchunks; ++ch) {
            // chunk geometry.  Plain input: columns [k0, k0+kc) of x.  Harmonic: dims [d0, d0+dcv) and harmonics [hs0, hs0+hc):
            // their dcv*hc sin columns (global column dd*Hn+h) followed by their dcv*hc cos columns (global column Hn*D + dd*Hn+h)
            const int dg = ch / nseg, hs0 = (ch - dg * nseg) * HC, hc = Hn > 0 ? imin(HC, Hn - hs0) : 0;
            const int d0 = dg * DC, dcv = Hn > 0 ? imin(DC, D - d0) : 0, half = dcv * hc;
            const int k0 = ch * KC, kc = Hn > 0 ? 2 * half : imin(KC, K - k0), kc4 = (kc + 3) >> 2;
            ex.phase([&](int tid) {
                if (Hn > 0) {
                    const bool pow2 = sm[L.flag] != 0.0f;
                    const int n8 = (hc + 7) >> 3;
                    for (int i = tid; i < nr * dcv * n8; i += nthr) {
                        const int hs = i % n8, rd = i / n8, dd = rd % dcv, r = rd / dcv;
                        const int h0 = 8 * hs, n = imin(8, hc - h0);
                        float sv[8], cv[8];
                        harmonics(sm[L.x + r * L.PD + d0 + dd], sm + L.freq, pow2, hs0 + h0, n, sv, cv);
                        float* es = sm + L.emb + r * PKC + dd * hc + h0;
                        for (int j = 0; j < n; ++j) { es[j] = sv[j]; es[half + j] = cv[j]; }
                    }
                    for (int i = tid; i < nr * (4 * kc4 - kc); i += nthr) {
                        const int r = i / (4 * kc4 - kc), c = kc + (i - r * (4 * kc4 - kc));
                        sm[L.emb + r * PKC + c] = 0.0f;
                    }
                    for (int i = tid; i < E * 4 * kc4; i += nthr) {
                        const int e = i / (4 * kc4), c = i - e * 4 * kc4;
                        const int cs = c < half ? c : c - half;
                        const int col = (c < half ? 0 : Hn * D) + d0 * Hn + (hc == Hn ? cs : (cs / hc) * Hn + hs0 + cs % hc);
                        sm[L.w + e * PKC + c] = c < kc ? a.w.w[(size_t)e * K + col] : 0.0f;
                    }
                } else {
                    for (int i = tid; i < nr * 4 * kc4; i += nthr) {
                        const int r = i / (4 * kc4), c = i - r * 4 * kc4;
                        sm[L.emb + r * PKC + c] = c < kc ? sm[L.x + r * L.PD + k0 + c] : 0.0f;
                    }
                    for (int i = tid; i < E * 4 * kc4; i += nthr) {
                        const int e = i / (4 * kc4), c = i - e * 4 * kc4;
                        sm[L.w + e * PKC + c] = c < kc ? a.w.w[(size_t)e * K + k0 + c] : 0.0f;
                    }
                }
            });
            ex.phase([&](int tid) {
                const int ks = tid / tiles, tl = tid - ks * tiles;
                if (ks < ksplit && tiles <= nthr) {
                    const int rt = tl / n_ct, ct = tl - rt * n_ct;
                    const float* ap[4];
                    const float* bp[4];
                    MMX_UNROLL
                    for (int i = 0; i < 4; ++i) ap[i] = sm + L.emb + imin(rt + i * n_rt, nr - 1) * PKC;
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j) bp[j] = sm + L.w + imin(ct + j * n_ct, E - 1) * PKC;
                    EncFwdRegs& rg = regs[tid];
                    for (int q = ks; q < kc4; q += ksplit) {
                        f4 av[4], bv[4];
                        MMX_UNROLL
                        for (int i = 0; i < 4; ++i) av[i] = ld4(ap[i] + 4 * q);
                        MMX_UNROLL
                        for (int j = 0; j < 4; ++j) bv[j] = ld4(bp[j] + 4 * q);
                        MMX_UNROLL
                        for (int i = 0; i < 4; ++i)
                            MMX_UNROLL
                            for (int j = 0; j < 4; ++j) {
                                rg.acc[i][j] = fmaf(av[i].x, bv[j].x, rg.acc[i][j]);
                                rg.acc[i][j] = fmaf(av[i].y, bv[j].y, rg.acc[i][j]);
                                rg.acc[i][j] = fmaf(av[i].z, bv[j].z, rg.acc[i][j]);
                                rg.acc[i][j] = fmaf(av[i].w, bv[j].w, rg.acc[i][j]);
                            }
                    }
                }
            });
        }
        ex.phase([&](int tid) {   // combine the K-split partial tiles
            const int ks = tid / tiles, tl = tid - ks * tiles;
            if (ks < ksplit && tiles <= nthr) {
                const int rt = tl / n_ct, ct = tl - rt * n_ct;
                EncFwdRegs& rg = regs[tid];
                MMX_UNROLL
                for (int i = 0; i < 4; ++i) {
                    const int r = rt + i * n_rt;
                    if (r < nr) {
                        MMX_UNROLL
                        for (int j = 0; j < 4; ++j) {
                            const int e = ct + j * n_ct;
                            if (e < E) smem_add(sm + L.m + r * PE + e, rg.acc[i][j]);
                        }
                    }
                }
            }
        });
        ex.phase([&](int tid) {
            for (int i = tid; i < nr * E; i += nthr) {
                const int r = i / E, e = i - r * E;
                const float mv = sm[L.m + r * PE + e] + sm[L.b + e];
                a.m[(size_t)(row0 + r) * E + e] = mv;
                const int b = (row0 + r) / T, t = (row0 + r) - b * T;
                for (int c = 0; c < C; ++c) a.y[((size_t)(b * C + c) * T + t) * E + e] = fmaf(mv, sm[L.wc + c], sm[L.bc + c]);
            }
        });
    }
}

// ------------------------------------------------------------------------------------------
// encoder backward, stage 1:  dm[r][e] = sum_c dy[b][c][t][e] wc[c];  dwc[c] += sum dy*m;  dbc[c] += sum dy;
//                             (with_db) db[e] += sum_r dm[r][e]
// ------------------------------------------------------------------------------------------
struct EncBwd1Dims { int B, T, E, C, R, with_db; };
struct EncBwd1Smem { int PE, dm, wc, a_wc, a_bc, a_b, total; };
MMX_HD EncBwd1Smem enc_bwd1_smem(const EncBwd1Dims& d) {
    EncBwd1Smem L; L.PE = pitch_of(d.E);
    int o = 0;
    auto take = [&](int n) { int r = o; o += round_up(n, 4); return r; };
    L.dm = take(d.R * L.PE); L.wc = take(8); L.a_wc = take(8); L.a_bc = take(8); L.a_b = take(d.E);
    L.total = o;
    return L;
}
struct EncBwd1Args { EncBwd1Dims d; const float* wc; const float* m; const float* dy; float* dm; float *g_wc, *g_bc, *g_b; };

MMX_D void enc_bwd1_body(Exec& ex, const EncBwd1Args& a) {
    const EncBwd1Dims& d = a.d;
    const EncBwd1Smem L = enc_bwd1_smem(d);
    float* sm = ex.smem;
    const int nthr = ex.nthr, E = d.E, C = d.C, T = d.T, R = d.R, PE = L.PE;
    const int rows = d.B * T;
    ex.phase([&](int tid) {
        for (int i = tid; i < 8; i += nthr) { sm[L.wc + i] = i < C ? a.wc[i] : 0.0f; sm[L.a_wc + i] = 0.0f; sm[L.a_bc + i] = 0.0f; }
        zero_vec(tid, nthr, sm + L.a_b, E);
    });
    const int ntiles = (rows + R - 1) / R;
    for (int tile = ex.bid; tile < ntiles; tile += ex.nblk) {
        const int row0 = tile * R, nr = imin(R, rows - row0);
        ex.phase([&](int tid) {
            float lw[8], lb[8];
            MMX_UNROLL
            for (int c = 0; c < 8; ++c) { lw[c] = 0.0f; lb[c] = 0.0f; }
            for (int i = tid; i < nr * E; i += nthr) {
                const int r = i / E, e = i - r * E;
                const int b = (row0 + r) / T, t = (row0 + r) - b * T;
                const float mv = a.m[(size_t)(row0 + r) * E + e];
                float dmv = 0.0f;
                MMX_UNROLL
                for (int c = 0; c < 8; ++c)
                    if (c < C) {
                        const float g = a.dy[((size_t)(b * C + c) * T + t) * E + e];
                        dmv = fmaf(g, sm[L.wc + c], dmv);
                        lw[c] = fmaf(g, mv, lw[c]); lb[c] += g;
                    }
                sm[L.dm + r * PE + e] = dmv;
                a.dm[(size_t)(row0 + r) * E + e] = dmv;
            }
            MMX_UNROLL
            for (int c = 0; c < 8; ++c)
                if (c < C) { smem_add(sm + L.a_wc + c, lw[c]); smem_add(sm + L.a_bc + c, lb[c]); }
        });
        if (d.with_db)
            ex.phase([&](int tid) {
                const int nsl = imax(1, nthr / E);
                for (int it = tid; it < E * nsl; it += nthr) {
                    const int sl = it / E, e = it - sl * E;
                    float s = 0.0f;
                    for (int r = sl; r < nr; r += nsl) s += sm[L.dm + r * PE + e];
                    smem_add(sm + L.a_b + e, s);
                }
            });
    }
    ex.phase([&](int tid) {
        for (int c = tid; c < C; c += nthr) { red_add(a.g_wc + c, sm[L.a_wc + c]); red_add(a.g_bc + c, sm[L.a_bc + c]); }
        if (d.with_db)
            for (int e = tid; e < E; e += nthr) red_add(a.g_b + e, sm[L.a_b + e]);
    });
}

// ------------------------------------------------------------------------------------------
// encoder backward, stage 2 (harmonic embedding only).  A CTA owns one input dimension dd and HC
// harmonics [h0, h0+HC): the sin columns dd*Hn+h and the cos columns Hn*D+dd*Hn+h of embed_mlp.weight.
// It sweeps ALL frames, regenerating its slice of the embedding, and accumulates
//     dW[e][col] += sum_r dm[r][e] emb[r][col]                 (thread-owned register tiles)
//     dx[r][dd]  += sum_h f[h] (cos(a) demb_sin - sin(a) demb_cos),   demb = dm W[:, cols]
// ------------------------------------------------------------------------------------------
struct EncBwd2Dims { int B, T, D, E, Hn, HC, R, need_dx; };
struct EncBwd2Smem { int PE, P2, dm, emb, w, cont, x, freq, flag, total; };
MMX_HD EncBwd2Smem enc_bwd2_smem(const EncBwd2Dims& d) {
    EncBwd2Smem L; L.PE = pitch_of(d.E); L.P2 = pitch_of(2 * d.HC);
    int o = 0;
    auto take = [&](int n) { int r = o; o += round_up(n, 4); return r; };
    L.dm = take(d.R * L.PE); L.emb = take(d.R * L.P2); L.w = take(d.E * L.P2); L.cont = take(d.R * L.P2);
    L.x = take(d.R); L.freq = take(d.Hn); L.flag = take(4);
    L.total = o;
    return L;
}
struct EncBwd2Args { EncBwd2Dims d; const float *freq, *w; const float* x; const float* dm; float* g_w; float* dx; };
struct EncBwd2Regs { float acc[4][4]; };

MMX_D void enc_bwd2_body(Exec& ex, const EncBwd2Args& a) {
    const EncBwd2Dims& d = a.d;
    const EncBwd2Smem L = enc_bwd2_smem(d);
    float* sm = ex.smem;
    const int nthr = ex.nthr, D = d.D, E = d.E, Hn = d.Hn, HC = d.HC, R = d.R, PE = L.PE, P2 = L.P2;
    const int rows = d.B * d.T, K = 2 * Hn * D;
    const int nseg = (Hn + HC - 1) / HC;
    const int w_nt = (2 * HC + 3) >> 2, w_tiles = ((E + 3) >> 2) * w_nt;   // dW slice [E][2*HC]
    PerThread<EncBwd2Regs> regs(ex);
    for (int grp = ex.bid; grp < D * nseg; grp += ex.nblk) {
        const int dd = grp / nseg, h0 = (grp - dd * nseg) * HC, hc = imin(HC, Hn - h0);
        const int col_s = dd * Hn + h0, col_c = Hn * D + dd * Hn + h0;
        ex.phase([&](int tid) {
            for (int i = tid; i < E * P2; i += nthr) {
                const int e = i / P2, c = i - e * P2;
                float v = 0.0f;
                if (c < HC) { if (c < hc) v = a.w[(size_t)e * K + col_s + c]; }
                else if (c < 2 * HC) { if (c - HC < hc) v = a.w[(size_t)e * K + col_c + c - HC]; }
                sm[L.w + i] = v;
            }
            for (int i = tid; i < Hn; i += nthr) sm[L.freq + i] = a.freq[i];
            if (tid == 0) sm[L.flag] = (float)freq_is_pow2_ladder(a.freq, Hn);
            EncBwd2Regs& rg = regs[tid];
            MMX_UNROLL
            for (int i = 0; i < 4; ++i)
                MMX_UNROLL
                for (int j = 0; j < 4; ++j) rg.acc[i][j] = 0.0f;
        });
        for (int row0 = 0; row0 < rows; row0 += R) {
            const int nr = imin(R, rows - row0);
            ex.phase([&](int tid) {
                load_tile(tid, nthr, sm + L.dm, a.dm + (size_t)row0 * E, nr, E, PE);
                const bool pow2 = sm[L.flag] != 0.0f;
                const int nsub = (HC + 7) >> 3;
                for (int i = tid; i < nr * nsub; i += nthr) {
                    const int r = i / nsub, sub = i - r * nsub;
                    const int hh = 8 * sub, n = imax(0, imin(8, hc - hh));      // harmonics h0+hh .. of this CTA's segment
                    float sv[8], cv[8];
                    if (n > 0) harmonics(a.x[(size_t)(row0 + r) * D + dd], sm + L.freq, pow2, h0 + hh, n, sv, cv);
                    for (int j = 0; j < imin(8, HC - hh); ++j) {
                        sm[L.emb + r * P2 + hh + j] = j < n ? sv[j] : 0.0f;
                        sm[L.emb + r * P2 + HC + hh + j] = j < n ? cv[j] : 0.0f;
                    }
                }
                for (int i = tid; i < nr * (P2 - 2 * HC); i += nthr) {
                    const int r = i / (P2 - 2 * HC), c = 2 * HC + (i - r * (P2 - 2 * HC));
                    sm[L.emb + r * P2 + c] = 0.0f;
                }
            });
            ex.phase([&](int tid) {
                if (tid < w_tiles) gemm_tn_acc4x4(regs[tid].acc, tid, w_nt, sm + L.dm, PE, sm + L.emb, P2, nr);
                if (d.need_dx)
                    gemm_nn<4>(tid, nthr, sm + L.dm, PE, sm + L.w, P2, nr, 2 * HC, E, [&](int m, int n, float v) {
                        // d sin(a)/da = cos(a), d cos(a)/da = -sin(a); da/dx = f
                        const float fr = sm[L.freq + imin(h0 + (n < HC ? n : n - HC), Hn - 1)];
                        const float c = n < HC ? v * sm[L.emb + m * P2 + n + HC] * fr : -v * sm[L.emb + m * P2 + n - HC] * fr;
                        sm[L.cont + m * P2 + n] = c;
                    });
            });
            if (d.need_dx)
                ex.phase([&](int tid) {
                    for (int r = tid; r < nr; r += nthr) {
                        float s = 0.0f;
                        for (int c = 0; c < 2 * HC; ++c) s += sm[L.cont + r * P2 + c];
                        red_add(a.dx + (size_t)(row0 + r) * D + dd, s);
                    }
                });
        }
        ex.phase([&](int tid) {
            if (tid < w_tiles) {
                const int mt = tid / w_nt, nt = tid - mt * w_nt;
                MMX_UNROLL
                for (int i = 0; i < 4; ++i) {
                    const int e = 4 * mt + i;
                    if (e < E) {
                        MMX_UNROLL
                        for (int j = 0; j < 4; ++j) {
                            const int c = 4 * nt + j;
                            if (c < HC) { if (c < hc) red_add(a.g_w + (size_t)e * K + col_s + c, regs[tid].acc[i][j]); }
                            else if (c < 2 * HC) { if (c - HC < hc) red_add(a.g_w + (size_t)e * K + col_c + c - HC, regs[tid].acc[i][j]); }
                        }
                    }
                }
            }
        });
    }
}

// ==========================================================================================
// ConvMixer head                                              conv_mixer_model.py:455-463
//   Q = LN(Y);  q[t][e] = sum_c wp[c] Q[c][t][e];  r[o][e] = sum_t Wt[o][t] q[t][e] + bt[o] sum_c wp[c] + bp
//   out[o][:] = Wf GELU(r[o][:]) + bf
// (project_channels and conv_out are both linear, so the channel mix is applied first: one time-mix
//  instead of C.)
// ==========================================================================================
struct ConvHeadDims {
    int B, C, T, To, E, D, S;
    int EC;       // chunked plan (conv_head_*_chunked_body): embedding columns per chunk, a multiple of 4; 0 for the resident plan
};
struct ConvHeadW { float *ln_g, *ln_b, *wt, *bt, *wp, *bp, *wf, *bf; };
struct ConvHeadSmem {
    int PE, PD, R, ln_g, ln_b, wt, bt, wp, wf, bf, part, part2, mean, rstd, bY, bQ, bR, bG, bO;
    int a_lng, a_lnb, a_bf, a_bt, a_wp, a_bp, a_wt, total;
};
MMX_HD ConvHeadSmem conv_head_smem(const ConvHeadDims& d, bool bwd) {
    ConvHeadSmem L; L.PE = pitch_of(d.E); L.PD = pitch_of(d.D); L.R = d.S * d.C * d.T;
    int o = 0;
    auto take = [&](int n) { int r = o; o += round_up(n, 4); return r; };
    L.ln_g = take(d.E); L.ln_b = take(d.E); L.wt = take(d.To * d.T); L.bt = take(d.To); L.wp = take(8 + 4);
    L.wf = take(d.D * L.PE); L.bf = take(d.D);
    const int nred = imax(L.R, d.S * d.To) * kParts;
    L.part = take(nred); L.part2 = take(nred); L.mean = take(L.R); L.rstd = take(L.R);
    L.bY = take(L.R * L.PE);
    L.bQ = take(d.S * d.T * L.PE);
    L.bG = take(d.S * d.To * L.PE);
    if (bwd) {
        L.bR = take(d.S * d.To * L.PE);
        L.bO = take(d.S * d.To * L.PD);
        L.a_lng = take(d.E); L.a_lnb = take(d.E); L.a_bf = take(d.D); L.a_bt = take(d.To); L.a_wp = take(8); L.a_bp = take(4);
        L.a_wt = take(d.To * d.T);
    } else { L.bR = L.bO = L.a_lng = L.a_lnb = L.a_bf = L.a_bt = L.a_wp = L.a_bp = L.a_wt = -1; }
    L.total = o;
    return L;
}

// small parameters of the head, and (resident plan) all of Wf; the chunked plan stages Wf one chunk at a time
template <class Layout>
MMX_D void conv_head_stage(int tid, int nthr, float* sm, const Layout& L, const ConvHeadDims& d, const ConvHeadW& w) {
    copy_vec(tid, nthr, sm + L.ln_g, w.ln_g, d.E); copy_vec(tid, nthr, sm + L.ln_b, w.ln_b, d.E);
    copy_vec(tid, nthr, sm + L.wt, w.wt, d.To * d.T); copy_vec(tid, nthr, sm + L.bt, w.bt, d.To);
    for (int i = tid; i < 8; i += nthr) sm[L.wp + i] = i < d.C ? w.wp[i] : 0.0f;
    if (tid == 0) {
        float sw = 0.0f;
        for (int c = 0; c < d.C; ++c) sw += w.wp[c];
        sm[L.wp + 8] = sw;          // sum_c wp[c]
        sm[L.wp + 9] = w.bp[0];
    }
    if (d.EC == 0) stage_matrix(tid, nthr, sm + L.wf, w.wf, d.D, d.E, L.PE);
    copy_vec(tid, nthr, sm + L.bf, w.bf, d.D);
}

// q (channel-mixed LN output) and r (pre-GELU) / g = GELU(r) of the tile; pad columns of bG are zeroed
template <class ExecT>
MMX_D void conv_head_forward_phases(ExecT& ex, float* sm, const ConvHeadSmem& L, const ConvHeadDims& d, int ns, bool keep_r) {
    const int nthr = ex.nthr, C = d.C, T = d.T, To = d.To, E = d.E, PE = L.PE;
    ex.phase([&](int tid) {
        for (int i = tid; i < ns * T * E; i += nthr) {
            const int st = i / E, e = i - st * E, s = st / T, t = st - s * T;
            float acc = 0.0f;
            for (int c = 0; c < C; ++c) {
                const int r = (s * C + c) * T + t;
                const float qv = (sm[L.bY + r * PE + e] - sm[L.mean + r]) * sm[L.rstd + r] * sm[L.ln_g + e] + sm[L.ln_b + e];
                acc = fmaf(sm[L.wp + c], qv, acc);
            }
            sm[L.bQ + st * PE + e] = acc;
        }
        for (int i = tid; i < ns * To * (PE - E); i += nthr) {
            const int r = i / (PE - E), c = E + (i - r * (PE - E));
            sm[L.bG + r * PE + c] = 0.0f;
            if (keep_r) sm[L.bR + r * PE + c] = 0.0f;
        }
        for (int i = tid; i < ns * T * (PE - E); i += nthr) {
            const int r = i / (PE - E), c = E + (i - r * (PE - E));
            sm[L.bQ + r * PE + c] = 0.0f;
        }
    });
    ex.phase([&](int tid) {
        for (int i = tid; i < ns * To * E; i += nthr) {
            const int so = i / E, e = i - so * E, s = so / To, o = so - s * To;
            float acc = fmaf(sm[L.bt + o], sm[L.wp + 8], sm[L.wp + 9]);
            for (int t = 0; t < T; ++t) acc = fmaf(sm[L.wt + o * T + t], sm[L.bQ + (s * T + t) * PE + e], acc);
            if (keep_r) sm[L.bR + so * PE + e] = acc;
            sm[L.bG + so * PE + e] = act_fwd<ACT_GELU>(acc);
        }
    });
}

struct ConvHeadFwdArgs { ConvHeadDims d; ConvHeadW w; const float* y; float* out; };

MMX_D void conv_head_fwd_body(Exec& ex, const ConvHeadFwdArgs& a) {
    const ConvHeadDims& d = a.d;
    const ConvHeadSmem L = conv_head_smem(d, false);
    float* sm = ex.smem;
    const int nthr = ex.nthr, C = d.C, T = d.T, To = d.To, E = d.E, D = d.D, S = d.S, PE = L.PE;
    ex.phase([&](int tid) { conv_head_stage(tid, nthr, sm, L, d, a.w); });
    const int ntiles = (d.B + S - 1) / S;
    for (int tile = ex.bid; tile < ntiles; tile += ex.nblk) {
        const long long seq0 = (long long)tile * S;
        const int ns = imin(S, d.B - (int)seq0), nr = ns * C * T;
        ex.phase([&](int tid) { load_tile(tid, nthr, sm + L.bY, a.y + (size_t)seq0 * C * T * E, nr, E, PE); });
        ln_stats_phases(ex, sm, L.part, L.part2, L.mean, L.rstd, sm + L.bY, PE, nr, E);
        conv_head_forward_phases(ex, sm, L, d, ns, false);
        ex.phase([&](int tid) {
            float* og = a.out + (size_t)seq0 * To * D;
            gemm_nt<4, 4>(tid, nthr, sm + L.bG, PE, sm + L.wf, PE, ns * To, D, E, [&](int m, int n, float v) {
                og[(size_t)m * D + n] = v + sm[L.bf + n];
            });
        });
    }
}

struct ConvHeadBwdArgs { ConvHeadDims d; ConvHeadW w; ConvHeadW g; const float* y; const float* dout; float* dy; };
template <int WT>
struct ConvHeadBwdRegs { float dWf[WT][4][4]; float dWt[4][4]; };

template <int WT>
MMX_D void conv_head_bwd_body(Exec& ex, const ConvHeadBwdArgs& a) {
    const ConvHeadDims& d = a.d;
    const ConvHeadSmem L = conv_head_smem(d, true);
    float* sm = ex.smem;
    const int nthr = ex.nthr, C = d.C, T = d.T, To = d.To, E = d.E, D = d.D, S = d.S, PE = L.PE, PD = L.PD;
    const float invE = 1.0f / (float)E;
    const int f_nt = (E + 3) >> 2, f_tiles = ((D + 3) >> 2) * f_nt;       // dWf [D][E]
    const bool persist = f_tiles <= nthr * WT;
    const int t_nt = (T + 3) >> 2, t_tiles = ((To + 3) >> 2) * t_nt;      // dWt [To][T]
    const int n_slices = imax(1, nthr / t_tiles);
    PerThread<ConvHeadBwdRegs<WT>> regs(ex);
    ex.phase([&](int tid) {
        conv_head_stage(tid, nthr, sm, L, d, a.w);
        zero_vec(tid, nthr, sm + L.a_lng, E); zero_vec(tid, nthr, sm + L.a_lnb, E);
        zero_vec(tid, nthr, sm + L.a_bf, D); zero_vec(tid, nthr, sm + L.a_bt, To);
        zero_vec(tid, nthr, sm + L.a_wp, 8); zero_vec(tid, nthr, sm + L.a_bp, 4); zero_vec(tid, nthr, sm + L.a_wt, To * T);
        ConvHeadBwdRegs<WT>& rg = regs[tid];
        MMX_UNROLL
        for (int w = 0; w < WT; ++w)
            MMX_UNROLL
            for (int i = 0; i < 4; ++i)
                MMX_UNROLL
                for (int j = 0; j < 4; ++j) rg.dWf[w][i][j] = 0.0f;
        MMX_UNROLL
        for (int i = 0; i < 4; ++i)
            MMX_UNROLL
            for (int j = 0; j < 4; ++j) rg.dWt[i][j] = 0.0f;
    });
    const int ntiles = (d.B + S - 1) / S;
    for (int tile = ex.bid; tile < ntiles; tile += ex.nblk) {
        const long long seq0 = (long long)tile * S;
        const int ns = imin(S, d.B - (int)seq0), nr = ns * C * T, no = ns * To;
        ex.phase([&](int tid) {
            load_tile(tid, nthr, sm + L.bY, a.y + (size_t)seq0 * C * T * E, nr, E, PE);
            load_tile(tid, nthr, sm + L.bO, a.dout + (size_t)seq0 * To * D, no, D, PD);
        });
        ln_stats_phases(ex, sm, L.part, L.part2, L.mean, L.rstd, sm + L.bY, PE, nr, E);
        conv_head_forward_phases(ex, sm, L, d, ns, true);
        // dbf, dWf[dd][e] += sum_rows dout[row][dd] g[row][e]
        ex.phase([&](int tid) {
            for (int n = tid; n < D; n += nthr) {
                float s = 0.0f;
                for (int r = 0; r < no; ++r) s += sm[L.bO + r * PD + n];
                sm[L.a_bf + n] += s;
            }
            ConvHeadBwdRegs<WT>& rg = regs[tid];
            if (persist) {
                MMX_UNROLL
                for (int w = 0; w < WT; ++w) {
                    const int t = tid + w * nthr;
                    if (t < f_tiles) gemm_tn_acc4x4(rg.dWf[w], t, f_nt, sm + L.bO, PD, sm + L.bG, PE, no);
                }
            } else {
                for (int t = tid; t < f_tiles; t += nthr) {
                    float acc[4][4] = {};
                    gemm_tn_acc4x4(acc, t, f_nt, sm + L.bO, PD, sm + L.bG, PE, no);
                    flush_acc4x4(acc, t, f_nt, a.g.wf, E, D, E);
                }
            }
        });
        // dr = (dout Wf) * gelu'(r)   -> bR in place
        ex.phase([&](int tid) {
            gemm_nn<4>(tid, nthr, sm + L.bO, PD, sm + L.wf, PE, no, E, D, [&](int m, int n, float v) {
                float ga;
                sm[L.bR + m * PE + n] = v * act_fwd_grad<ACT_GELU>(sm[L.bR + m * PE + n], &ga);
            });
        });
        // row sums of dr (-> dbp, dbt, the bias part of dwp);  dWt[o][t] += sum_{s,e} dr[s,o,e] q[s,t,e]
        ex.phase([&](int tid) {
            for (int i = tid; i < no * kParts; i += nthr) sm[L.part + i] = row_part_sum(sm + L.bR + (i / kParts) * PE, E, i % kParts);
            ConvHeadBwdRegs<WT>& rg = regs[tid];
            const int slice = tid / t_tiles, otile = tid - slice * t_tiles;
            if (slice < n_slices) {
                const int E4 = (E + 3) >> 2;
                const int mt = otile / t_nt, nt = otile - mt * t_nt;
                for (int s = slice; s < ns; s += n_slices) {
                    const float* A = sm + L.bR + (s * To) * PE;
                    const float* Bm = sm + L.bQ + (s * T) * PE;
                    for (int q = 0; q < E4; ++q) {
                        f4 av[4], bv[4];
                        MMX_UNROLL
                        for (int i = 0; i < 4; ++i) av[i] = ld4(A + imin(4 * mt + i, To - 1) * PE + 4 * q);
                        MMX_UNROLL
                        for (int j = 0; j < 4; ++j) bv[j] = ld4(Bm + imin(4 * nt + j, T - 1) * PE + 4 * q);
                        MMX_UNROLL
                        for (int i = 0; i < 4; ++i)
                            MMX_UNROLL
                            for (int j = 0; j < 4; ++j)
                                rg.dWt[i][j] += (av[i].x * bv[j].x + av[i].y * bv[j].y) + (av[i].z * bv[j].z + av[i].w * bv[j].w);
                    }
                }
            }
        });
        // dq[s][t][e] = sum_o Wt[o][t] dr[s][o][e]  -> bQ (q is dead after dWt) ... needs q for nothing else
        ex.phase([&](int tid) {
            for (int o = tid; o < To; o += nthr) {      // drsum[o] over the tile's sequences
                float s_ = 0.0f;
                for (int s = 0; s < ns; ++s) s_ += sum_parts(sm + L.part + (s * To + o) * kParts);
                sm[L.a_bt + o] += s_ * sm[L.wp + 8];
                smem_add(sm + L.a_bp, s_);
                // bias part of dwp[c]: sum_o bt[o] drsum[o]  (same for every c) accumulated in a_bp[1]
                smem_add(sm + L.a_bp + 1, s_ * sm[L.bt + o]);
            }
        });
        ex.phase([&](int tid) {
            for (int i = tid; i < ns * T * E; i += nthr) {
                const int st = i / E, e = i - st * E, s = st / T, t = st - s * T;
                float acc = 0.0f;
                for (int o = 0; o < To; ++o) acc = fmaf(sm[L.wt + o * T + t], sm[L.bR + (s * To + o) * PE + e], acc);
                sm[L.bQ + st * PE + e] = acc;
            }
        });
        // dwp[c] += sum Q dq ;  LN backward with dQ[s,c,t,e] = wp[c] dq[s,t,e]
        ex.phase([&](int tid) {
            const int nsl = imax(1, nthr / E);
            for (int it = tid; it < E * nsl; it += nthr) {
                const int sl = it / E, e = it - sl * E;
                float sg = 0.0f, sb = 0.0f;
                for (int r = sl; r < nr; r += nsl) {
                    const int sc = r / T, t = r - sc * T, s = sc / C, c = sc - s * C;
                    const float dn = sm[L.wp + c] * sm[L.bQ + (s * T + t) * PE + e];
                    const float xh = (sm[L.bY + r * PE + e] - sm[L.mean + r]) * sm[L.rstd + r];
                    sg = fmaf(dn, xh, sg); sb += dn;
                }
                smem_add(sm + L.a_lng + e, sg); smem_add(sm + L.a_lnb + e, sb);
            }
            for (int i = tid; i < nr * kParts; i += nthr) {
                const int r = i / kParts, p = i - r * kParts;
                const int sc = r / T, t = r - sc * T, s = sc / C, c = sc - s * C;
                const float mu = sm[L.mean + r], rs = sm[L.rstd + r], wpc = sm[L.wp + c];
                const float* dq = sm + L.bQ + (s * T + t) * PE;
                const float* yr = sm + L.bY + r * PE;
                float m1 = 0.0f, m2 = 0.0f, qd = 0.0f;
                for (int h = 4 * p; h < E; h += 4 * kParts) {
                    const int n = imin(4, E - h);
                    for (int k = 0; k < n; ++k) {
                        const float xh = (yr[h + k] - mu) * rs;
                        const float dxh = wpc * dq[h + k] * sm[L.ln_g + h + k];
                        m1 += dxh; m2 = fmaf(dxh, xh, m2);
                        qd = fmaf(fmaf(xh, sm[L.ln_g + h + k], sm[L.ln_b + h + k]), dq[h + k], qd);
                    }
                }
                sm[L.part + i] = m1; sm[L.part2 + i] = m2;
                smem_add(sm + L.a_wp + c, qd);
            }
        });
        ex.phase([&](int tid) {
            float* dyg = a.dy + (size_t)seq0 * C * T * E;
            for (int i = tid; i < nr * E; i += nthr) {
                const int r = i / E, e = i - r * E;
                const int sc = r / T, t = r - sc * T, s = sc / C, c = sc - s * C;
                const float mu = sm[L.mean + r], rs = sm[L.rstd + r];
                const float m1 = sum_parts(sm + L.part + r * kParts) * invE, m2 = sum_parts(sm + L.part2 + r * kParts) * invE;
                const float dxh = sm[L.wp + c] * sm[L.bQ + (s * T + t) * PE + e] * sm[L.ln_g + e];
                const float xh = (sm[L.bY + r * PE + e] - mu) * rs;
                dyg[(size_t)r * E + e] = rs * (dxh - m1 - xh * m2);
            }
        });
    }
    ex.phase([&](int tid) {
        ConvHeadBwdRegs<WT>& rg = regs[tid];
        if (persist) {
            MMX_UNROLL
            for (int w = 0; w < WT; ++w) {
                const int t = tid + w * nthr;
                if (t < f_tiles) flush_acc4x4(rg.dWf[w], t, f_nt, a.g.wf, E, D, E);
            }
        }
        const int slice = tid / t_tiles, otile = tid - slice * t_tiles;
        if (slice < n_slices) smem_add_acc4x4(rg.dWt, otile, t_nt, sm + L.a_wt, T, To, T);    // combine the CTA's K-split slices
        for (int e = tid; e < E; e += nthr) { red_add(a.g.ln_g + e, sm[L.a_lng + e]); red_add(a.g.ln_b + e, sm[L.a_lnb + e]); }
        for (int n = tid; n < D; n += nthr) red_add(a.g.bf + n, sm[L.a_bf + n]);
        for (int o = tid; o < To; o += nthr) red_add(a.g.bt + o, sm[L.a_bt + o]);
        for (int c = tid; c < C; c += nthr) red_add(a.g.wp + c, sm[L.a_wp + c] + sm[L.a_bp + 1]);
        if (tid == 0) red_add(a.g.bp, sm[L.a_bp]);
    });
    ex.phase([&](int tid) {
        for (int i = tid; i < To * T; i += nthr) red_add(a.g.wt + i, sm[L.a_wt + i]);
    });
}

// ------------------------------------------------------------------------------------------
// Chunked head plan, for the shapes whose resident tile (all of Wf [D][E] plus the tile's Y, q, r, g rows) does not fit
// shared memory.  Only the LayerNorm statistics and the fc_out contraction span E; everything else is elementwise in e.
// A tile takes its row statistics from Y in global memory, then walks the embedding in chunks of EC columns: it stages
// Wf[:, chunk], forms q, r and g of the chunk (reading Y from global memory) and accumulates out over the chunks.
// The backward makes the same sweep and accumulates every parameter gradient and the two per-row LayerNorm sums m1, m2
// that dy needs; it keeps the tile's dq [S*T][E] so that dy is one elementwise pass after the sweep.  The CTA's partial
// dWf [D][E] stays in shared memory for the whole persistent loop and is flushed once, as the resident plan does with
// registers.
// ------------------------------------------------------------------------------------------
struct ConvHeadChunkSmem {
    int PC, PE, PD, R, ln_g, ln_b, wt, bt, wp, bf, wf, part, part2, mean, rstd, bQ, bG, bO;
    int bR, dq, pm1, pm2, a_wf, a_lng, a_lnb, a_bf, a_bt, a_wp, a_bp, a_wt, total;
};
MMX_HD ConvHeadChunkSmem conv_head_chunk_smem(const ConvHeadDims& d, bool bwd) {
    ConvHeadChunkSmem L; L.PC = pitch_of(d.EC); L.PE = pitch_of(d.E); L.PD = pitch_of(d.D); L.R = d.S * d.C * d.T;
    const int no = d.S * d.To;
    int o = 0;
    auto take = [&](int n) { int r = o; o += round_up(n, 4); return r; };
    L.ln_g = take(d.E); L.ln_b = take(d.E); L.wt = take(d.To * d.T); L.bt = take(d.To); L.wp = take(8 + 4); L.bf = take(d.D);
    L.wf = take(d.D * L.PC);
    const int nred = imax(L.R, no) * kParts;
    L.part = take(nred); L.part2 = take(nred); L.mean = take(L.R); L.rstd = take(L.R);
    L.bQ = take(d.S * d.T * L.PC); L.bG = take(no * L.PC); L.bO = take(no * L.PD);   // bO: out accumulator (fwd), dout (bwd)
    if (bwd) {
        L.bR = take(no * L.PC); L.dq = take(d.S * d.T * L.PE); L.pm1 = take(L.R * kParts); L.pm2 = take(L.R * kParts);
        L.a_wf = take(d.D * d.E); L.a_lng = take(d.E); L.a_lnb = take(d.E); L.a_bf = take(d.D); L.a_bt = take(d.To);
        L.a_wp = take(8); L.a_bp = take(4); L.a_wt = take(d.To * d.T);
    } else { L.bR = L.dq = L.pm1 = L.pm2 = L.a_wf = L.a_lng = L.a_lnb = L.a_bf = L.a_bt = L.a_wp = L.a_bp = L.a_wt = -1; }
    L.total = o;
    return L;
}

// Wf[:, e0:e0+ec) -> wf [D][PC] and q of the chunk -> bQ [ns*T][PC] (Y from global); pad columns zeroed
MMX_D void conv_head_chunk_stage_q(int tid, int nthr, float* sm, const ConvHeadChunkSmem& L, const ConvHeadDims& d,
                                   const ConvHeadW& w, const float* yg, int ns, int e0, int ec) {
    const int C = d.C, T = d.T, E = d.E, PC = L.PC;
    for (int i = tid; i < d.D * PC; i += nthr) {
        const int n = i / PC, j = i - n * PC;
        sm[L.wf + i] = j < ec ? w.wf[(size_t)n * E + e0 + j] : 0.0f;
    }
    for (int i = tid; i < ns * T * PC; i += nthr) {
        const int st = i / PC, j = i - st * PC, s = st / T, t = st - s * T, e = e0 + j;
        float acc = 0.0f;
        if (j < ec)
            for (int c = 0; c < C; ++c) {
                const int r = (s * C + c) * T + t;
                const float qv = (yg[(size_t)r * E + e] - sm[L.mean + r]) * sm[L.rstd + r] * sm[L.ln_g + e] + sm[L.ln_b + e];
                acc = fmaf(sm[L.wp + c], qv, acc);
            }
        sm[L.bQ + i] = acc;
    }
}

// r (pre-GELU, bwd only -> bR) and g = GELU(r) -> bG of the chunk; pad columns zeroed
MMX_D void conv_head_chunk_rg(int tid, int nthr, float* sm, const ConvHeadChunkSmem& L, const ConvHeadDims& d, int ns, int ec, bool keep_r) {
    const int T = d.T, To = d.To, PC = L.PC;
    for (int i = tid; i < ns * To * PC; i += nthr) {
        const int so = i / PC, j = i - so * PC, s = so / To, o = so - s * To;
        float acc = 0.0f, g = 0.0f;
        if (j < ec) {
            acc = fmaf(sm[L.bt + o], sm[L.wp + 8], sm[L.wp + 9]);
            for (int t = 0; t < T; ++t) acc = fmaf(sm[L.wt + o * T + t], sm[L.bQ + (s * T + t) * PC + j], acc);
            g = act_fwd<ACT_GELU>(acc);
        }
        if (keep_r) sm[L.bR + i] = acc;
        sm[L.bG + i] = g;
    }
}

MMX_D void conv_head_fwd_chunked_body(Exec& ex, const ConvHeadFwdArgs& a) {
    const ConvHeadDims& d = a.d;
    const ConvHeadChunkSmem L = conv_head_chunk_smem(d, false);
    float* sm = ex.smem;
    const int nthr = ex.nthr, C = d.C, T = d.T, To = d.To, E = d.E, D = d.D, S = d.S, PC = L.PC, PD = L.PD;
    ex.phase([&](int tid) { conv_head_stage(tid, nthr, sm, L, d, a.w); });
    const int ntiles = (d.B + S - 1) / S;
    for (int tile = ex.bid; tile < ntiles; tile += ex.nblk) {
        const long long seq0 = (long long)tile * S;
        const int ns = imin(S, d.B - (int)seq0), nr = ns * C * T, no = ns * To;
        const float* yg = a.y + (size_t)seq0 * C * T * E;
        ln_stats_phases(ex, sm, L.part, L.part2, L.mean, L.rstd, yg, E, nr, E);
        for (int e0 = 0; e0 < E; e0 += d.EC) {
            const int ec = imin(d.EC, E - e0);
            ex.phase([&](int tid) {
                if (e0 == 0) zero_vec(tid, nthr, sm + L.bO, no * PD);
                conv_head_chunk_stage_q(tid, nthr, sm, L, d, a.w, yg, ns, e0, ec);
            });
            ex.phase([&](int tid) { conv_head_chunk_rg(tid, nthr, sm, L, d, ns, ec, false); });
            ex.phase([&](int tid) {
                gemm_nt<4, 4>(tid, nthr, sm + L.bG, PC, sm + L.wf, PC, no, D, ec, [&](int m, int n, float v) { sm[L.bO + m * PD + n] += v; });
            });
        }
        ex.phase([&](int tid) {
            float* og = a.out + (size_t)seq0 * To * D;
            for (int i = tid; i < no * D; i += nthr) {
                const int m = i / D, n = i - m * D;
                og[i] = sm[L.bO + m * PD + n] + sm[L.bf + n];
            }
        });
    }
}

struct ConvHeadChunkBwdRegs { float dWt[4][4]; };

MMX_D void conv_head_bwd_chunked_body(Exec& ex, const ConvHeadBwdArgs& a) {
    const ConvHeadDims& d = a.d;
    const ConvHeadChunkSmem L = conv_head_chunk_smem(d, true);
    float* sm = ex.smem;
    const int nthr = ex.nthr, C = d.C, T = d.T, To = d.To, E = d.E, D = d.D, S = d.S, PC = L.PC, PE = L.PE, PD = L.PD;
    const float invE = 1.0f / (float)E;
    const int t_nt = (T + 3) >> 2, t_tiles = ((To + 3) >> 2) * t_nt;      // dWt [To][T]
    const int n_slices = imax(1, nthr / t_tiles);
    PerThread<ConvHeadChunkBwdRegs> regs(ex);
    ex.phase([&](int tid) {
        conv_head_stage(tid, nthr, sm, L, d, a.w);
        zero_vec(tid, nthr, sm + L.a_wf, D * E);
        zero_vec(tid, nthr, sm + L.a_lng, E); zero_vec(tid, nthr, sm + L.a_lnb, E);
        zero_vec(tid, nthr, sm + L.a_bf, D); zero_vec(tid, nthr, sm + L.a_bt, To);
        zero_vec(tid, nthr, sm + L.a_wp, 8); zero_vec(tid, nthr, sm + L.a_bp, 4); zero_vec(tid, nthr, sm + L.a_wt, To * T);
        ConvHeadChunkBwdRegs& rg = regs[tid];
        MMX_UNROLL
        for (int i = 0; i < 4; ++i)
            MMX_UNROLL
            for (int j = 0; j < 4; ++j) rg.dWt[i][j] = 0.0f;
    });
    const int ntiles = (d.B + S - 1) / S;
    for (int tile = ex.bid; tile < ntiles; tile += ex.nblk) {
        const long long seq0 = (long long)tile * S;
        const int ns = imin(S, d.B - (int)seq0), nr = ns * C * T, no = ns * To;
        const float* yg = a.y + (size_t)seq0 * C * T * E;
        ex.phase([&](int tid) {
            load_tile(tid, nthr, sm + L.bO, a.dout + (size_t)seq0 * To * D, no, D, PD);
            zero_vec(tid, nthr, sm + L.pm1, nr * kParts); zero_vec(tid, nthr, sm + L.pm2, nr * kParts);
        });
        ln_stats_phases(ex, sm, L.part, L.part2, L.mean, L.rstd, yg, E, nr, E);
        for (int e0 = 0; e0 < E; e0 += d.EC) {
            const int ec = imin(d.EC, E - e0);
            ex.phase([&](int tid) {
                if (e0 == 0)
                    for (int n = tid; n < D; n += nthr) {
                        float s = 0.0f;
                        for (int r = 0; r < no; ++r) s += sm[L.bO + r * PD + n];
                        sm[L.a_bf + n] += s;
                    }
                conv_head_chunk_stage_q(tid, nthr, sm, L, d, a.w, yg, ns, e0, ec);
            });
            ex.phase([&](int tid) { conv_head_chunk_rg(tid, nthr, sm, L, d, ns, ec, true); });
            // dWf[n][e0+j] += sum_rows dout[row][n] g[row][j];  dr = (dout Wf) * gelu'(r) -> bR in place
            ex.phase([&](int tid) {
                const int f_nt = (ec + 3) >> 2, f_tiles = ((D + 3) >> 2) * f_nt;
                for (int t = tid; t < f_tiles; t += nthr) {
                    float acc[4][4] = {};
                    gemm_tn_acc4x4(acc, t, f_nt, sm + L.bO, PD, sm + L.bG, PC, no);
                    const int mt = t / f_nt, nt = t - mt * f_nt;
                    MMX_UNROLL
                    for (int i = 0; i < 4; ++i)
                        MMX_UNROLL
                        for (int j = 0; j < 4; ++j)
                            if (4 * mt + i < D && 4 * nt + j < ec) sm[L.a_wf + (4 * mt + i) * E + e0 + 4 * nt + j] += acc[i][j];
                }
                gemm_nn<4>(tid, nthr, sm + L.bO, PD, sm + L.wf, PC, no, ec, D, [&](int m, int n, float v) {
                    float ga;
                    sm[L.bR + m * PC + n] = v * act_fwd_grad<ACT_GELU>(sm[L.bR + m * PC + n], &ga);
                });
            });
            // row sums of dr (-> dbp, dbt, the bias part of dwp);  dWt[o][t] += sum_{s,e} dr[s,o,e] q[s,t,e]
            ex.phase([&](int tid) {
                for (int i = tid; i < no * kParts; i += nthr) sm[L.part + i] = row_part_sum(sm + L.bR + (i / kParts) * PC, ec, i % kParts);
                ConvHeadChunkBwdRegs& rg = regs[tid];
                const int slice = tid / t_tiles, otile = tid - slice * t_tiles;
                if (slice < n_slices) {
                    const int E4 = (ec + 3) >> 2;
                    const int mt = otile / t_nt, nt = otile - mt * t_nt;
                    for (int s = slice; s < ns; s += n_slices) {
                        const float* A = sm + L.bR + (s * To) * PC;
                        const float* Bm = sm + L.bQ + (s * T) * PC;
                        for (int q = 0; q < E4; ++q) {
                            f4 av[4], bv[4];
                            MMX_UNROLL
                            for (int i = 0; i < 4; ++i) av[i] = ld4(A + imin(4 * mt + i, To - 1) * PC + 4 * q);
                            MMX_UNROLL
                            for (int j = 0; j < 4; ++j) bv[j] = ld4(Bm + imin(4 * nt + j, T - 1) * PC + 4 * q);
                            MMX_UNROLL
                            for (int i = 0; i < 4; ++i)
                                MMX_UNROLL
                                for (int j = 0; j < 4; ++j)
                                    rg.dWt[i][j] += (av[i].x * bv[j].x + av[i].y * bv[j].y) + (av[i].z * bv[j].z + av[i].w * bv[j].w);
                        }
                    }
                }
            });
            // drsum[o] over the tile's sequences -> dbt, dbp, bias part of dwp;  dq[s][t][e0+j] = sum_o Wt[o][t] dr[s][o][j]
            ex.phase([&](int tid) {
                for (int o = tid; o < To; o += nthr) {
                    float s_ = 0.0f;
                    for (int s = 0; s < ns; ++s) s_ += sum_parts(sm + L.part + (s * To + o) * kParts);
                    sm[L.a_bt + o] += s_ * sm[L.wp + 8];
                    smem_add(sm + L.a_bp, s_);
                    smem_add(sm + L.a_bp + 1, s_ * sm[L.bt + o]);
                }
                for (int i = tid; i < ns * T * ec; i += nthr) {
                    const int st = i / ec, j = i - st * ec, s = st / T, t = st - s * T;
                    float acc = 0.0f;
                    for (int o = 0; o < To; ++o) acc = fmaf(sm[L.wt + o * T + t], sm[L.bR + (s * To + o) * PC + j], acc);
                    sm[L.dq + st * PE + e0 + j] = acc;
                }
            });
            // dgamma, dbeta of the chunk's columns; dwp[c] += sum Q dq; the chunk's share of the LN sums m1, m2 of every row
            ex.phase([&](int tid) {
                const int nsl = imax(1, nthr / ec);
                for (int it = tid; it < ec * nsl; it += nthr) {
                    const int sl = it / ec, e = e0 + (it - sl * ec);
                    float sg = 0.0f, sb = 0.0f;
                    for (int r = sl; r < nr; r += nsl) {
                        const int sc = r / T, t = r - sc * T, s = sc / C, c = sc - s * C;
                        const float dn = sm[L.wp + c] * sm[L.dq + (s * T + t) * PE + e];
                        const float xh = (yg[(size_t)r * E + e] - sm[L.mean + r]) * sm[L.rstd + r];
                        sg = fmaf(dn, xh, sg); sb += dn;
                    }
                    smem_add(sm + L.a_lng + e, sg); smem_add(sm + L.a_lnb + e, sb);
                }
                for (int i = tid; i < nr * kParts; i += nthr) {
                    const int r = i / kParts, p = i - r * kParts;
                    const int sc = r / T, t = r - sc * T, s = sc / C, c = sc - s * C;
                    const float mu = sm[L.mean + r], rs = sm[L.rstd + r], wpc = sm[L.wp + c];
                    const float* dq = sm + L.dq + (s * T + t) * PE + e0;
                    const float* yr = yg + (size_t)r * E + e0;
                    const float* lg = sm + L.ln_g + e0;
                    const float* lb = sm + L.ln_b + e0;
                    float m1 = 0.0f, m2 = 0.0f, qd = 0.0f;
                    for (int h = 4 * p; h < ec; h += 4 * kParts) {
                        const int n = imin(4, ec - h);
                        for (int k = 0; k < n; ++k) {
                            const float xh = (yr[h + k] - mu) * rs;
                            const float dxh = wpc * dq[h + k] * lg[h + k];
                            m1 += dxh; m2 = fmaf(dxh, xh, m2);
                            qd = fmaf(fmaf(xh, lg[h + k], lb[h + k]), dq[h + k], qd);
                        }
                    }
                    sm[L.pm1 + i] += m1; sm[L.pm2 + i] += m2;
                    smem_add(sm + L.a_wp + c, qd);
                }
            });
        }
        ex.phase([&](int tid) {
            float* dyg = a.dy + (size_t)seq0 * C * T * E;
            for (int i = tid; i < nr * E; i += nthr) {
                const int r = i / E, e = i - r * E;
                const int sc = r / T, t = r - sc * T, s = sc / C, c = sc - s * C;
                const float mu = sm[L.mean + r], rs = sm[L.rstd + r];
                const float m1 = sum_parts(sm + L.pm1 + r * kParts) * invE, m2 = sum_parts(sm + L.pm2 + r * kParts) * invE;
                const float dxh = sm[L.wp + c] * sm[L.dq + (s * T + t) * PE + e] * sm[L.ln_g + e];
                const float xh = (yg[i] - mu) * rs;
                dyg[i] = rs * (dxh - m1 - xh * m2);
            }
        });
    }
    ex.phase([&](int tid) {
        for (int i = tid; i < D * E; i += nthr) red_add(a.g.wf + i, sm[L.a_wf + i]);
        const int slice = tid / t_tiles, otile = tid - slice * t_tiles;
        if (slice < n_slices) smem_add_acc4x4(regs[tid].dWt, otile, t_nt, sm + L.a_wt, T, To, T);    // combine the CTA's K-split slices
        for (int e = tid; e < E; e += nthr) { red_add(a.g.ln_g + e, sm[L.a_lng + e]); red_add(a.g.ln_b + e, sm[L.a_lnb + e]); }
        for (int n = tid; n < D; n += nthr) red_add(a.g.bf + n, sm[L.a_bf + n]);
        for (int o = tid; o < To; o += nthr) red_add(a.g.bt + o, sm[L.a_bt + o]);
        for (int c = tid; c < C; c += nthr) red_add(a.g.wp + c, sm[L.a_wp + c] + sm[L.a_bp + 1]);
        if (tid == 0) red_add(a.g.bp, sm[L.a_bp]);
    });
    ex.phase([&](int tid) {
        for (int i = tid; i < To * T; i += nthr) red_add(a.g.wt + i, sm[L.a_wt + i]);
    });
}

}  // namespace mmx

namespace mmx {

// ==========================================================================================
// BatchNorm halves (regularization == -1): the two passes that are NOT convolutions.
//   apply (forward) :  R = act(Z)*scale[c] + shift[c] ;  y = x + SE(R)
//   bwd1 (backward) :  gate, ds from SE backward with dgate = sum dy*R ;  dR = dy*gate + ds/(C*E) ;
//                      sums[c] += sum dR ;  sums[C+c] += sum dR*xhat  (xhat = act(Z)*xs[c] + xo[c]) ;  gd[b][t] = (gate, ds)
// Both stream x / Z / dy from global (elementwise + per-(sequence, frame) reductions; mean squeeze only).
// ==========================================================================================
struct BnPassDims { int B, C, T, E, rr, S, use_se, act; };
struct BnPassSmem { int se1, se2, part, part2, pool, gate, z, dq, dz, ds, a_se1, a_se2, a_sum, bn, total; };
MMX_HD BnPassSmem bn_pass_smem(const BnPassDims& d) {
    BnPassSmem L;
    const int rr = imax(d.rr, 1), ST = d.S * d.T;
    int o = 0;
    auto take = [&](int n) { int r = o; o += round_up(n, 4); return r; };
    L.se1 = take(rr * d.T); L.se2 = take(d.T * rr);
    L.part = take(ST * d.C * kParts); L.part2 = take(ST * d.C * kParts);     // per (sequence, channel, frame) row
    L.pool = take(ST); L.gate = take(ST); L.z = take(d.S * rr); L.dq = take(ST); L.dz = take(d.S * rr); L.ds = take(ST);
    L.a_se1 = take(rr * d.T); L.a_se2 = take(d.T * rr); L.a_sum = take(16); L.bn = take(32);
    L.total = o;
    return L;
}
struct BnPassArgs {
    BnPassDims d;
    const float *se1, *se2;   // SE parameters (null without SE)
    float *g_se1, *g_se2;     // SE gradient accumulators (bwd1)
    const float* bn;          // [scale | shift | xs | xo][C]
    const float* x;           // apply: half input
    const float* z;           // pre-activation from the statistics pass
    const float* dy;          // bwd1: upstream gradient
    float* y;                 // apply: half output
    float* gd;                // bwd1: [B,T,2] (gate, ds)
    double* sums;             // bwd1: [sum dR | sum dR*xhat][C]
};

template <int ACT>
MMX_D void bn_apply_fwd_body(Exec& ex, const BnPassArgs& a) {
    const BnPassDims& d = a.d;
    const BnPassSmem L = bn_pass_smem(d);
    float* sm = ex.smem;
    const int nthr = ex.nthr, C = d.C, T = d.T, E = d.E, S = d.S, rr = d.rr;
    const float invCE = 1.0f / (float)(C * E);
    ex.phase([&](int tid) {
        if (d.use_se) { copy_vec(tid, nthr, sm + L.se1, a.se1, rr * T); copy_vec(tid, nthr, sm + L.se2, a.se2, T * rr); }
        for (int i = tid; i < 4 * C; i += nthr) sm[L.bn + (i / C) * 8 + i % C] = a.bn[i];
    });
    const int ntiles = (d.B + S - 1) / S;
    for (int tile = ex.bid; tile < ntiles; tile += ex.nblk) {
        const long long seq0 = (long long)tile * S;
        const int ns = imin(S, d.B - (int)seq0), nr = ns * C * T;
        const float* xg = a.x + (size_t)seq0 * C * T * E;
        const float* zg = a.z + (size_t)seq0 * C * T * E;
        float* yg = a.y + (size_t)seq0 * C * T * E;
        if (d.use_se) {
            ex.phase([&](int tid) {      // row partials: every thread busy (rows = sequences x channels x frames)
                for (int i = tid; i < nr * kParts; i += nthr) {
                    const int r = i / kParts, p = i - r * kParts, c = (r / T) % C;
                    const float sc = sm[L.bn + c], sh = sm[L.bn + 8 + c];
                    const float* zr = zg + (size_t)r * E;
                    float acc = 0.0f;
                    for (int h = 4 * p; h < E; h += 4 * kParts) {
                        const int n = imin(4, E - h);
                        for (int k = 0; k < n; ++k) acc += fmaf(act_fwd<ACT>(zr[h + k]), sc, sh);
                    }
                    sm[L.part + i] = acc;
                }
            });
            ex.phase([&](int tid) {
                for (int st = tid; st < ns * T; st += nthr) {
                    const int s = st / T, t = st - s * T;
                    float acc = 0.0f;
                    for (int c = 0; c < C; ++c) acc += sum_parts(sm + L.part + ((s * C + c) * T + t) * kParts);
                    sm[L.pool + st] = acc * invCE;
                }
            });
            ex.phase([&](int tid) {
                for (int st = tid; st < ns * T; st += nthr) {
                    const int s = st / T, t = st - s * T;
                    sm[L.gate + st] = se_excite(sm + L.se1, sm + L.se2, sm + L.pool + s * T, T, rr, t, nullptr);
                }
            });
        }
        ex.phase([&](int tid) {
            for (int i = tid; i < nr * E; i += nthr) {
                const int r = i / E, sc_ = r / T, t = r - sc_ * T, s = sc_ / C, c = sc_ - s * C;
                const float g = d.use_se ? sm[L.gate + s * T + t] : 1.0f;
                const float rv = fmaf(act_fwd<ACT>(zg[i]), sm[L.bn + c], sm[L.bn + 8 + c]);
                yg[i] = fmaf(g, rv, xg[i]);
            }
        });
    }
}

template <int ACT>
MMX_D void bn_bwd1_body(Exec& ex, const BnPassArgs& a) {
    const BnPassDims& d = a.d;
    const BnPassSmem L = bn_pass_smem(d);
    float* sm = ex.smem;
    const int nthr = ex.nthr, C = d.C, T = d.T, E = d.E, S = d.S, rr = d.rr;
    const float invCE = 1.0f / (float)(C * E);
    ex.phase([&](int tid) {
        if (d.use_se) {
            copy_vec(tid, nthr, sm + L.se1, a.se1, rr * T); copy_vec(tid, nthr, sm + L.se2, a.se2, T * rr);
            zero_vec(tid, nthr, sm + L.a_se1, rr * T); zero_vec(tid, nthr, sm + L.a_se2, T * rr);
        }
        for (int i = tid; i < 16; i += nthr) sm[L.a_sum + i] = 0.0f;
        for (int i = tid; i < 4 * C; i += nthr) sm[L.bn + (i / C) * 8 + i % C] = a.bn[i];
    });
    const int ntiles = (d.B + S - 1) / S;
    for (int tile = ex.bid; tile < ntiles; tile += ex.nblk) {
        const long long seq0 = (long long)tile * S;
        const int ns = imin(S, d.B - (int)seq0);
        const float* zg = a.z + (size_t)seq0 * C * T * E;
        const float* dyg = a.dy + (size_t)seq0 * C * T * E;
        if (d.use_se) {
            ex.phase([&](int tid) {      // squeeze of R and dgate = sum dy*R: row partials
                for (int i = tid; i < ns * C * T * kParts; i += nthr) {
                    const int r = i / kParts, p = i - r * kParts, c = (r / T) % C;
                    const float sc = sm[L.bn + c], sh = sm[L.bn + 8 + c];
                    const size_t off = (size_t)r * E;
                    float acc = 0.0f, dg = 0.0f;
                    for (int h = 4 * p; h < E; h += 4 * kParts) {
                        const int n = imin(4, E - h);
                        for (int k = 0; k < n; ++k) {
                            const float rv = fmaf(act_fwd<ACT>(zg[off + h + k]), sc, sh);
                            acc += rv; dg = fmaf(dyg[off + h + k], rv, dg);
                        }
                    }
                    sm[L.part + i] = acc; sm[L.part2 + i] = dg;
                }
            });
            ex.phase([&](int tid) {
                for (int st = tid; st < ns * T; st += nthr) {
                    const int s = st / T, t = st - s * T;
                    float acc = 0.0f, dg = 0.0f;
                    for (int c = 0; c < C; ++c) {
                        acc += sum_parts(sm + L.part + ((s * C + c) * T + t) * kParts);
                        dg += sum_parts(sm + L.part2 + ((s * C + c) * T + t) * kParts);
                    }
                    sm[L.pool + st] = acc * invCE;
                    sm[L.dq + st] = dg;
                }
            });
            ex.phase([&](int tid) {
                for (int st = tid; st < ns * T; st += nthr) {
                    const int s = st / T, t = st - s * T;
                    sm[L.gate + st] = se_excite(sm + L.se1, sm + L.se2, sm + L.pool + s * T, T, rr, t, sm + L.z + s * rr);
                }
            });
            se_bwd_phases(ex, sm, T, rr, ns, L.se1, L.se2, L.dq, L.dz, L.gate, L.pool, L.z, L.ds, L.a_se1, L.a_se2);
        }
        // dR = dy*gate + ds/(C*E): per-channel sums of dR and dR*xhat; (gate, ds) saved for pass 2
        ex.phase([&](int tid) {
            for (int st = tid; st < ns * T; st += nthr) {
                a.gd[((size_t)seq0 * T + st) * 2] = d.use_se ? sm[L.gate + st] : 1.0f;
                a.gd[((size_t)seq0 * T + st) * 2 + 1] = d.use_se ? sm[L.ds + st] : 0.0f;
            }
            for (int i = tid; i < ns * C * T * kParts; i += nthr) {
                const int r = i / kParts, p = i - r * kParts, sc_ = r / T, t = r - sc_ * T, s = sc_ / C, c = sc_ - s * C;
                const float g = d.use_se ? sm[L.gate + s * T + t] : 1.0f;
                const float dsv = d.use_se ? sm[L.ds + s * T + t] * invCE : 0.0f;
                const float xs = sm[L.bn + 16 + c], xo = sm[L.bn + 24 + c];
                const size_t off = (size_t)r * E;
                float s1 = 0.0f, s2 = 0.0f;
                for (int h = 4 * p; h < E; h += 4 * kParts) {
                    const int n = imin(4, E - h);
                    for (int k = 0; k < n; ++k) {
                        const float dr_ = fmaf(dyg[off + h + k], g, dsv);
                        const float xh = fmaf(act_fwd<ACT>(zg[off + h + k]), xs, xo);
                        s1 += dr_; s2 = fmaf(dr_, xh, s2);
                    }
                }
                smem_add(sm + L.a_sum + c, s1); smem_add(sm + L.a_sum + 8 + c, s2);
            }
        });
    }
    ex.phase([&](int tid) {
        for (int i = tid; i < C; i += nthr) {
            red_add_f64(a.sums + i, (double)sm[L.a_sum + i]);
            red_add_f64(a.sums + C + i, (double)sm[L.a_sum + 8 + i]);
        }
        if (d.use_se)
            for (int i = tid; i < T * rr; i += nthr) { red_add(a.g_se1 + i, sm[L.a_se1 + i]); red_add(a.g_se2 + i, sm[L.a_se2 + i]); }
    });
}

}  // namespace mmx
