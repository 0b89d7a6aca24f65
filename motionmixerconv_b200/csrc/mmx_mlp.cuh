// Fused MotionMixer (MlpMixer) kernels: embed, mixer block forward / backward, head.
//
// Reference arithmetic: h36m/mlp_mixer.py  SELayer :30-34, MlpBlock :87-96,
// MixerBlock.forward :138-164, MlpMixer.forward :325-337 (restated in SURVEY.md Appendix A.1
// and in oracle/mixer_np.py, which is the checker for these kernels).
//
// One CTA owns a tile of S whole sequences (R = S*T rows of the [B,T,H] activation) and keeps
// it resident in shared memory through every stage of the block; HBM sees one read of the
// block input and one write of the block output (forward), and block input + upstream
// gradient in, input gradient out (backward: the forward is recomputed in-kernel from the
// saved block input).  Weight gradients are accumulated in thread-owned registers / shared
// memory across the CTA's persistent loop over tiles and flushed once with RED.ADD.
#pragma once
#include "mmx_common.cuh"

namespace mmx {

constexpr int kParts = 8;   // partial sums per row / per (sequence, frame) in the reduction phases

// ------------------------------------------------------------------------------------------
// row reductions with kParts threads per row.  Part p handles quads p, p+kParts, ... of the row.
// ------------------------------------------------------------------------------------------
MMX_D float row_part_sum(const float* row, int W, int p) {
    float s = 0.0f;
    for (int h = 4 * p; h < W; h += 4 * kParts) {
        const int n = imin(4, W - h);
        for (int k = 0; k < n; ++k) s += row[h + k];
    }
    return s;
}
MMX_D float row_part_sqdev(const float* row, int W, float mu, int p) {
    float s = 0.0f;
    for (int h = 4 * p; h < W; h += 4 * kParts) {
        const int n = imin(4, W - h);
        for (int k = 0; k < n; ++k) { const float dv = row[h + k] - mu; s = fmaf(dv, dv, s); }
    }
    return s;
}
MMX_D float sum_parts(const float* p) {
    return ((p[0] + p[1]) + (p[2] + p[3])) + ((p[4] + p[5]) + (p[6] + p[7]));
}

// LayerNorm statistics (biased variance, two passes) of `nr` rows of width W -> sm[o_mean..], sm[o_rstd..]
template <class ExecT>
MMX_D void ln_stats_phases(ExecT& ex, float* sm, int o_part, int o_part2, int o_mean, int o_rstd,
                           const float* rows, int pitch, int nr, int W) {
    const int nthr = ex.nthr;
    ex.phase([&](int tid) {
        for (int i = tid; i < nr * kParts; i += nthr)
            sm[o_part + i] = row_part_sum(rows + (size_t)(i / kParts) * pitch, W, i % kParts);
    });
    ex.phase([&](int tid) {
        for (int i = tid; i < nr * kParts; i += nthr) {
            const int r = i / kParts, p = i - r * kParts;
            const float mu = sum_parts(sm + o_part + r * kParts) / (float)W;
            if (p == 0) sm[o_mean + r] = mu;
            sm[o_part2 + i] = row_part_sqdev(rows + (size_t)r * pitch, W, mu, p);
        }
    });
    ex.phase([&](int tid) {
        for (int r = tid; r < nr; r += nthr)
            sm[o_rstd + r] = 1.0f / sqrtf(sum_parts(sm + o_part2 + r * kParts) / (float)W + 1e-5f);
    });
}


struct MlpDims {
    int B, T, H, tok, ch, rr;  // rr = SE hidden width = T / r_se
    int S;                     // sequences per CTA tile
    int use_se, use_max;
    int training;
    int site_base;             // dropout site id of this block's first Dropout (block_index*4)
    int w_in_smem;             // 1: channel-MLP weights staged in shared memory, 0: read from global (needs H%4==0, ch%4==0)
};

struct MlpBlockW {            // parameter (or gradient) pointers of one MixerBlock, reference layouts
    float *ln1_g, *ln1_b;     // LN1.weight/bias                       [H]
    float *tw1, *tb1;         // mlp_block_token_mixing.fc1.weight/bias   [tok,T],[tok]
    float *tw2, *tb2;         // mlp_block_token_mixing.fc2.weight/bias   [T,tok],[T]
    float *ln2_g, *ln2_b;     // LN2.weight/bias                       [H]
    float *cw1, *cb1;         // mlp_block_channel_mixing.fc1.weight/bias [ch,H],[ch]
    float *cw2, *cb2;         // mlp_block_channel_mixing.fc2.weight/bias [H,ch],[H]
    float *se1, *se2;         // se.excitation.0.weight [rr,T], se.excitation.2.weight [T,rr]
};

// ------------------------------------------------------------------------------------------
// shared-memory layout (offsets in floats)
// ------------------------------------------------------------------------------------------
struct MlpBlockSmem {
    int PH, PC, R;
    // weights
    int ln1_g, ln1_b, ln2_g, ln2_b, tw1, tb1, tw2, tb2, cw1, cb1, cw2, cb2, se1, se2;
    // per-row / per-sequence small arrays
    int mean1, rstd1, mean2, rstd2, pool1, gate1, pool2, gate2, z1, z2, amax1, amax2;
    int dq, dz, ds1, ds2;
    int part, part2;                   // kParts partial sums per row (row reductions with several threads per row)
    // gradient accumulators owned by single threads (backward only)
    int a_ln1g, a_ln1b, a_ln2g, a_ln2b, a_cb1, a_cb2, a_se1, a_se2, a_tb1, a_tb2;
    // activation tiles
    int bX, bD, bYt, scratch;
    int bX1, bA, bY2, bU, bG;          // channel-half view of scratch
    int bN1, bdN1, tG, tdU;            // token-half view of scratch
    int total;
};

MMX_HD MlpBlockSmem mlp_block_smem(const MlpDims& d, bool bwd) {
    MlpBlockSmem L;
    const int T = d.T, H = d.H, tok = d.tok, ch = d.ch, rr = imax(d.rr, 1), S = d.S;
    L.PH = pitch_of(H);
    L.PC = pitch_of(ch);
    L.R = S * T;
    int o = 0;
    auto take = [&](int n) { int r = o; o += round_up(n, 4); return r; };
    L.ln1_g = take(H); L.ln1_b = take(H); L.ln2_g = take(H); L.ln2_b = take(H);
    L.tw1 = take(tok * T); L.tb1 = take(tok); L.tw2 = take(T * tok); L.tb2 = take(T);
    L.cb1 = take(ch); L.cb2 = take(H);
    L.se1 = take(rr * T); L.se2 = take(T * rr);
    if (d.w_in_smem) { L.cw1 = take(ch * L.PH); L.cw2 = take(H * L.PC); } else { L.cw1 = L.cw2 = -1; }
    L.mean1 = take(L.R); L.rstd1 = take(L.R); L.mean2 = take(L.R); L.rstd2 = take(L.R);
    L.pool1 = take(L.R); L.gate1 = take(L.R); L.pool2 = take(L.R); L.gate2 = take(L.R);
    L.z1 = take(S * rr); L.z2 = take(S * rr); L.amax1 = take(L.R); L.amax2 = take(L.R);
    L.dq = take(L.R); L.dz = take(S * rr); L.ds1 = take(L.R); L.ds2 = take(L.R);
    L.part = take(L.R * kParts); L.part2 = take(L.R * kParts);
    if (bwd) {
        L.a_ln1g = take(H); L.a_ln1b = take(H); L.a_ln2g = take(H); L.a_ln2b = take(H);
        L.a_cb1 = take(ch); L.a_cb2 = take(H); L.a_se1 = take(rr * T); L.a_se2 = take(T * rr);
        L.a_tb1 = take(tok); L.a_tb2 = take(T);
    } else {
        L.a_ln1g = L.a_ln1b = L.a_ln2g = L.a_ln2b = L.a_cb1 = L.a_cb2 = L.a_se1 = L.a_se2 = L.a_tb1 = L.a_tb2 = -1;
    }
    const int RH = L.R * L.PH, RC = L.R * L.PC;
    L.bX = take(RH);
    if (bwd) { L.bD = take(RH); L.bYt = take(RH); } else { L.bD = L.bYt = -1; }
    L.scratch = o;
    // channel-half view
    int c = L.scratch;
    if (bwd) { L.bX1 = c; c += RH; } else { L.bX1 = L.bX; }
    L.bA = c; c += RH;
    if (bwd) { L.bY2 = c; c += RH; } else { L.bY2 = L.bA; }
    L.bG = c; c += RC;
    if (bwd) { L.bU = c; c += RC; } else { L.bU = -1; }
    int t = L.scratch;
    if (bwd) {
        L.bN1 = t; t += RH; L.bdN1 = t; t += RH;
        L.tG = t; t += S * tok * L.PH; L.tdU = t; t += S * tok * L.PH;
    } else { L.bN1 = L.bdN1 = L.tG = L.tdU = -1; }
    if (!bwd) L.bYt = L.bA;   // forward: token-mix output goes straight into bA
    L.total = imax(c, t);
    return L;
}

// ------------------------------------------------------------------------------------------
// shared phases
// ------------------------------------------------------------------------------------------
MMX_D void copy_vec(int tid, int nthr, float* dst, const float* src, int n) {
    for (int i = tid; i < n; i += nthr) dst[i] = src[i];
}
MMX_D void zero_vec(int tid, int nthr, float* dst, int n) {
    for (int i = tid; i < n; i += nthr) dst[i] = 0.0f;
}
// stage a row-major [rows][cols] global matrix into shared with pitch P, zero-filling the pad columns
MMX_D void stage_matrix(int tid, int nthr, float* dst, const float* src, int rows, int cols, int P) {
    for (int i = tid; i < rows * P; i += nthr) {
        const int r = i / P, c = i - r * P;
        dst[i] = c < cols ? src[(size_t)r * cols + c] : 0.0f;
    }
}
// load a tile of nr rows x W floats (contiguous in global) into a pitched shared tile, zero pad columns
MMX_D void load_tile(int tid, int nthr, float* dst, const float* src, int nr, int W, int P) {
    if ((W & 3) == 0) {
        const int W4 = W >> 2;
        for (int i = tid; i < nr * W4; i += nthr) {
            const int r = i / W4, q = i - r * W4;
            st4(dst + r * P + 4 * q, ld4(src + (size_t)r * W + 4 * q));
        }
    } else if ((((uintptr_t)src) & 15) == 0) {
        // rows are not 16-byte multiples, but the tile is one contiguous, aligned run: stream it as float4 and scatter
        const int total = nr * W, Q = total >> 2;
        for (int i = tid; i < Q; i += nthr) {
            const f4 v = ld4(src + 4 * i);
            int r = (4 * i) / W, c = 4 * i - r * W;
            dst[r * P + c] = v.x; if (++c == W) { c = 0; ++r; }
            dst[r * P + c] = v.y; if (++c == W) { c = 0; ++r; }
            dst[r * P + c] = v.z; if (++c == W) { c = 0; ++r; }
            dst[r * P + c] = v.w;
        }
        for (int i = 4 * Q + tid; i < total; i += nthr) { const int r = i / W, c = i - r * W; dst[r * P + c] = src[i]; }
    } else {
        for (int i = tid; i < nr * W; i += nthr) {
            const int r = i / W, c = i - r * W;
            dst[r * P + c] = src[(size_t)r * W + c];
        }
    }
    if (P > W)
        for (int i = tid; i < nr * (P - W); i += nthr) {
            const int r = i / (P - W), c = W + (i - r * (P - W));
            dst[r * P + c] = 0.0f;
        }
}
MMX_D void store_tile(int tid, int nthr, float* dst, const float* src, int nr, int W, int P) {
    if ((W & 3) == 0) {
        const int W4 = W >> 2;
        for (int i = tid; i < nr * W4; i += nthr) {
            const int r = i / W4, q = i - r * W4;
            st4(dst + (size_t)r * W + 4 * q, ld4(src + r * P + 4 * q));
        }
    } else if ((((uintptr_t)dst) & 15) == 0) {
        const int total = nr * W, Q = total >> 2;
        for (int i = tid; i < Q; i += nthr) {
            int r = (4 * i) / W, c = 4 * i - r * W;
            f4 v;
            v.x = src[r * P + c]; if (++c == W) { c = 0; ++r; }
            v.y = src[r * P + c]; if (++c == W) { c = 0; ++r; }
            v.z = src[r * P + c]; if (++c == W) { c = 0; ++r; }
            v.w = src[r * P + c];
            st4(dst + 4 * i, v);
        }
        for (int i = 4 * Q + tid; i < total; i += nthr) { const int r = i / W, c = i - r * W; dst[i] = src[r * P + c]; }
    } else {
        for (int i = tid; i < nr * W; i += nthr) {
            const int r = i / W, c = i - r * W;
            dst[(size_t)r * W + c] = src[r * P + c];
        }
    }
}

// SE squeeze of one row: mean or (first) max over the W valid columns
MMX_D void row_pool(const float* row, int W, int use_max, float* pool, float* amax) {
    if (use_max) {
        float m = row[0]; int am = 0;
        for (int h = 1; h < W; ++h) { float v = row[h]; if (v > m) { m = v; am = h; } }
        *pool = m; *amax = (float)am;
    } else {
        float s = 0.0f;
        const int W4 = (W + 3) >> 2;
        for (int q = 0; q < W4; ++q) { f4 v = ld4(row + 4 * q); s += (v.x + v.y) + (v.z + v.w); }
        *pool = s / (float)W;
    }
}

// SE squeeze of nr rows: mean via kParts partial sums per row (every thread busy), max via one thread per row
template <class ExecT>
MMX_D void row_pool_phases(ExecT& ex, float* sm, const float* rows, int pitch, int nr, int W, int use_max, int o_pool, int o_amax, int o_part) {
    const int nthr = ex.nthr;
    if (use_max) {
        ex.phase([&](int tid) {
            for (int r = tid; r < nr; r += nthr) row_pool(rows + (size_t)r * pitch, W, 1, sm + o_pool + r, sm + o_amax + r);
        });
        return;
    }
    ex.phase([&](int tid) {
        for (int i = tid; i < nr * kParts; i += nthr) sm[o_part + i] = row_part_sum(rows + (size_t)(i / kParts) * pitch, W, i % kParts);
    });
    ex.phase([&](int tid) {
        for (int r = tid; r < nr; r += nthr) sm[o_pool + r] = sum_parts(sm + o_part + r * kParts) / (float)W;
    });
}

// dot[r] = sum_h A[r][h] * B[r][h] for nr rows, kParts threads per row
template <class ExecT>
MMX_D void row_dot_phases(ExecT& ex, float* sm, const float* A, const float* Bm, int pitch, int nr, int W, int o_dot, int o_part) {
    const int nthr = ex.nthr;
    ex.phase([&](int tid) {
        for (int i = tid; i < nr * kParts; i += nthr) {
            const int r = i / kParts, p = i - r * kParts;
            const float* ar = A + (size_t)r * pitch;
            const float* br = Bm + (size_t)r * pitch;
            float s = 0.0f;
            for (int h = 4 * p; h < W; h += 4 * kParts) {
                const int n = imin(4, W - h);
                for (int k = 0; k < n; ++k) s = fmaf(ar[h + k], br[h + k], s);
            }
            sm[o_part + i] = s;
        }
    });
    ex.phase([&](int tid) {
        for (int r = tid; r < nr; r += nthr) sm[o_dot + r] = sum_parts(sm + o_part + r * kParts);
    });
}

// SE excitation for row r = (s,t): gate = sigmoid(S2[t,:] . relu(S1 . pool[s,:])); thread t==0 of the
// sequence also stores the pre-activation z[s,:] (needed by the backward)
MMX_D float se_excite(const float* se1, const float* se2, const float* pool_s, int T, int rr, int t, float* z_s) {
    float q = 0.0f;
    for (int j = 0; j < rr; ++j) {
        float z = 0.0f;
        for (int tt = 0; tt < T; ++tt) z = fmaf(se1[j * T + tt], pool_s[tt], z);
        if (t == 0 && z_s) z_s[j] = z;
        q = fmaf(se2[t * rr + j], fmaxf(z, 0.0f), q);
    }
    return sigmoidf_(q);
}

// token-mixing MLP of one (sequence, channel) pair, everything in registers.
//   n[t] = LN1(x)[t,h];  u[k] = b1[k] + sum_t W1[k,t] n[t];  g[k] = act(u[k]) * mask1;
//   y[t] = (b2[t] + sum_k W2[t,k] g[k]) * mask2
// TC/TOKC > 0: exact compile-time seq_len / tokens_mlp_dim (loops fully unrolled, arrays in registers).
// TC == 0: generic path, runtime bounds (T <= 32, tok <= 64), arrays indexed dynamically.
template <int TC> struct TDim { static constexpr int cap = TC > 0 ? TC : 32; };
template <int KC> struct KDim { static constexpr int cap = KC > 0 ? KC : 64; };

template <int ACT, int TC, int TOKC>
struct TokenMix {
    float n[TDim<TC>::cap], u[KDim<TOKC>::cap], g[KDim<TOKC>::cap], y[TDim<TC>::cap];
    MMX_D void fwd(const float* sm, const MlpBlockSmem& L, const MlpDims& d, const Dropout& dr,
                   int s, int h, long long seq0) {
        const int T = d.T, tok = d.tok;
        const float gam = sm[L.ln1_g + h], bet = sm[L.ln1_b + h];
        MMX_UNROLL
        for (int t = 0; t < (TC > 0 ? TC : T); ++t)
            {
                const int r = s * T + t;
                n[t] = (sm[L.bX + r * L.PH + h] - sm[L.mean1 + r]) * sm[L.rstd1 + r] * gam + bet;
            }
        const bool drop = d.training && dr.thresh != 0u;
        const unsigned long long pair = (unsigned long long)(seq0 + s) * d.H + h;
        MMX_UNROLL
        for (int k = 0; k < (TOKC > 0 ? TOKC : tok); ++k)
            {
                float a = sm[L.tb1 + k];
                MMX_UNROLL
                for (int t = 0; t < (TC > 0 ? TC : T); ++t)
                    a = fmaf(sm[L.tw1 + k * T + t], n[t], a);
                u[k] = a;
                float gv = act_fwd<ACT>(a);
                if (drop) gv *= dropout_scale(dr, d.site_base + 0, pair * tok + k);
                g[k] = gv;
            }
        MMX_UNROLL
        for (int t = 0; t < (TC > 0 ? TC : T); ++t)
            {
                float a = sm[L.tb2 + t];
                MMX_UNROLL
                for (int k = 0; k < (TOKC > 0 ? TOKC : tok); ++k)
                    a = fmaf(sm[L.tw2 + t * tok + k], g[k], a);
                if (drop) a *= dropout_scale(dr, d.site_base + 1, pair * T + t);
                y[t] = a;
            }
    }
};

struct MlpBlockFwdArgs {
    MlpDims d;
    Dropout dr;
    MlpBlockW w;
    const float* x;
    float* y;
};

MMX_D void mlp_stage_weights(int tid, int nthr, float* sm, const MlpBlockSmem& L, const MlpDims& d, const MlpBlockW& w) {
    const int T = d.T, H = d.H, tok = d.tok, ch = d.ch, rr = d.rr;
    copy_vec(tid, nthr, sm + L.ln1_g, w.ln1_g, H); copy_vec(tid, nthr, sm + L.ln1_b, w.ln1_b, H);
    copy_vec(tid, nthr, sm + L.ln2_g, w.ln2_g, H); copy_vec(tid, nthr, sm + L.ln2_b, w.ln2_b, H);
    copy_vec(tid, nthr, sm + L.tw1, w.tw1, tok * T); copy_vec(tid, nthr, sm + L.tb1, w.tb1, tok);
    copy_vec(tid, nthr, sm + L.tw2, w.tw2, T * tok); copy_vec(tid, nthr, sm + L.tb2, w.tb2, T);
    copy_vec(tid, nthr, sm + L.cb1, w.cb1, ch); copy_vec(tid, nthr, sm + L.cb2, w.cb2, H);
    if (d.use_se) { copy_vec(tid, nthr, sm + L.se1, w.se1, rr * T); copy_vec(tid, nthr, sm + L.se2, w.se2, T * rr); }
    if (d.w_in_smem) {
        stage_matrix(tid, nthr, sm + L.cw1, w.cw1, ch, H, L.PH);
        stage_matrix(tid, nthr, sm + L.cw2, w.cw2, H, ch, L.PC);
    }
}

// ------------------------------------------------------------------------------------------
// MixerBlock forward  (mlp_mixer.py:138-164)
// ------------------------------------------------------------------------------------------
template <int ACT, int TC, int TOKC>
MMX_D void mlp_block_fwd_body(Exec& ex, const MlpBlockFwdArgs& a) {
    const MlpDims& d = a.d;
    const MlpBlockSmem L = mlp_block_smem(d, false);
    float* sm = ex.smem;
    const int nthr = ex.nthr;
    const int T = d.T, H = d.H, ch = d.ch, rr = d.rr, S = d.S, PH = L.PH, PC = L.PC;
    const float* V1 = d.w_in_smem ? sm + L.cw1 : a.w.cw1;
    const float* V2 = d.w_in_smem ? sm + L.cw2 : a.w.cw2;
    const int ldv1 = d.w_in_smem ? PH : H, ldv2 = d.w_in_smem ? PC : ch;
    const Dropout dr = resolve_dropout(a.dr);
    const bool drop = d.training && dr.thresh != 0u;

    ex.phase([&](int tid) { mlp_stage_weights(tid, nthr, sm, L, d, a.w); });

    const int ntiles = (d.B + S - 1) / S;
    for (int tile = ex.bid; tile < ntiles; tile += ex.nblk) {
        const long long seq0 = (long long)tile * S;
        const int ns = imin(S, d.B - (int)seq0), nr = ns * T;
        const float* xg = a.x + (size_t)seq0 * T * H;
        float* yg = a.y + (size_t)seq0 * T * H;

        ex.phase([&](int tid) {
            load_tile(tid, nthr, sm + L.bX, xg, nr, H, PH);
            // pad columns of the GEMM A-operands must be finite zeros
            for (int i = tid; i < nr * (PH - H); i += nthr) { int r = i / (PH - H); sm[L.bA + r * PH + H + (i - r * (PH - H))] = 0.0f; }
            for (int i = tid; i < nr * (PC - ch); i += nthr) { int r = i / (PC - ch); sm[L.bG + r * PC + ch + (i - r * (PC - ch))] = 0.0f; }
        });
        ln_stats_phases(ex, sm, L.part, L.part2, L.mean1, L.rstd1, sm + L.bX, PH, nr, H);
        // token mixing: one thread per (sequence, channel)
        ex.phase([&](int tid) {
            TokenMix<ACT, TC, TOKC> tm;
            for (int p = tid; p < ns * H; p += nthr) {
                const int s = p / H, h = p - s * H;
                tm.fwd(sm, L, d, dr, s, h, seq0);
                MMX_UNROLL
                for (int t = 0; t < (TC > 0 ? TC : T); ++t)
                    sm[L.bA + (s * T + t) * PH + h] = tm.y[t];
            }
        });
        if (d.use_se) {
            row_pool_phases(ex, sm, sm + L.bA, PH, nr, H, d.use_max, L.pool1, L.amax1, L.part);
            ex.phase([&](int tid) {
                for (int r = tid; r < nr; r += nthr) {
                    const int s = r / T, t = r - s * T;
                    sm[L.gate1 + r] = se_excite(sm + L.se1, sm + L.se2, sm + L.pool1 + s * T, T, rr, t, nullptr);
                }
            });
        }
        // X1 = X + gate*Yt ; LN2 statistics
        ex.phase([&](int tid) {
            for (int i = tid; i < nr * H; i += nthr) {
                const int r = i / H, h = i - r * H;
                const float g = d.use_se ? sm[L.gate1 + r] : 1.0f;
                sm[L.bX + r * PH + h] = fmaf(g, sm[L.bA + r * PH + h], sm[L.bX + r * PH + h]);
            }
        });
        ln_stats_phases(ex, sm, L.part, L.part2, L.mean2, L.rstd2, sm + L.bX, PH, nr, H);
        ex.phase([&](int tid) {
            for (int i = tid; i < nr * H; i += nthr) {
                const int r = i / H, h = i - r * H;
                sm[L.bA + r * PH + h] = (sm[L.bX + r * PH + h] - sm[L.mean2 + r]) * sm[L.rstd2 + r] * sm[L.ln2_g + h] + sm[L.ln2_b + h];
            }
        });
        // channel mixing: U2 = N2 V1^T + c1 ; G2 = act(U2)
        ex.phase([&](int tid) {
            gemm_nt<4, 4>(tid, nthr, sm + L.bA, PH, V1, ldv1, nr, ch, H, [&](int m, int n, float v) {
                float gv = act_fwd<ACT>(v + sm[L.cb1 + n]);
                if (drop) gv *= dropout_scale(dr, d.site_base + 2, ((unsigned long long)seq0 * T + m) * ch + n);
                sm[L.bG + m * PC + n] = gv;
            });
        });
        ex.phase([&](int tid) {
            gemm_nt<4, 4>(tid, nthr, sm + L.bG, PC, V2, ldv2, nr, H, ch, [&](int m, int n, float v) {
                float yv = v + sm[L.cb2 + n];
                if (drop) yv *= dropout_scale(dr, d.site_base + 3, ((unsigned long long)seq0 * T + m) * H + n);
                sm[L.bA + m * PH + n] = yv;
            });
        });
        if (d.use_se) {
            row_pool_phases(ex, sm, sm + L.bA, PH, nr, H, d.use_max, L.pool2, L.amax2, L.part);
            ex.phase([&](int tid) {
                for (int r = tid; r < nr; r += nthr) {
                    const int s = r / T, t = r - s * T;
                    sm[L.gate2 + r] = se_excite(sm + L.se1, sm + L.se2, sm + L.pool2 + s * T, T, rr, t, nullptr);
                }
            });
        }
        // out = X1 + gate2 * Y2  (coalesced 128-bit stores)
        ex.phase([&](int tid) {
            if ((H & 3) == 0) {
                const int H4 = H >> 2;
                for (int i = tid; i < nr * H4; i += nthr) {
                    const int r = i / H4, q = i - r * H4;
                    const float g = d.use_se ? sm[L.gate2 + r] : 1.0f;
                    f4 xv = ld4(sm + L.bX + r * PH + 4 * q), yv = ld4(sm + L.bA + r * PH + 4 * q);
                    st4(yg + (size_t)r * H + 4 * q, make_f4(fmaf(g, yv.x, xv.x), fmaf(g, yv.y, xv.y), fmaf(g, yv.z, xv.z), fmaf(g, yv.w, xv.w)));
                }
            } else {
                for (int i = tid; i < nr * H; i += nthr) {
                    const int r = i / H, h = i - r * H;
                    const float g = d.use_se ? sm[L.gate2 + r] : 1.0f;
                    yg[(size_t)r * H + h] = fmaf(g, sm[L.bA + r * PH + h], sm[L.bX + r * PH + h]);
                }
            }
        });
    }
}

// ------------------------------------------------------------------------------------------
// MixerBlock backward (forward recomputed from the saved block input)
// ------------------------------------------------------------------------------------------
struct MlpBlockBwdArgs {
    MlpDims d;
    Dropout dr;
    MlpBlockW w;     // parameters
    MlpBlockW g;     // gradient accumulators (global, += via RED)
    const float* x;  // block input  [B,T,H]
    const float* dy; // dL/d(block output)
    float* dx;       // dL/d(block input)
};

template <int WT>
struct MlpBwdRegs {
    float dV1[WT][4][4];   // dL/d cw1 tiles  [ch][H]
    float dV2[WT][4][4];   // dL/d cw2 tiles  [H][ch]
    float dW1[4][4];       // dL/d tw1 tile   [tok][T]   (split-K slice)
    float dW2[4][4];       // dL/d tw2 tile   [T][tok]
};

// SE backward for one squeeze-excitation use.  Inputs (shared): dg[r] = sum_h dOut*Y (in L.dq),
// gate, pool, z.  Outputs: ds[r] (gradient w.r.t. the pooled value), a_se1/a_se2 accumulators.
template <class ExecT>
MMX_D void se_backward_phases(ExecT& ex, float* sm, const MlpBlockSmem& L, const MlpDims& d, int ns,
                              int o_gate, int o_pool, int o_z, int o_ds) {
    const int T = d.T, rr = d.rr, nthr = ex.nthr, nr = ns * T;
    ex.phase([&](int tid) {   // dq = dg * g * (1-g)
        for (int r = tid; r < nr; r += nthr) { const float g = sm[o_gate + r]; sm[L.dq + r] *= g * (1.0f - g); }
    });
    ex.phase([&](int tid) {   // dz[s,j] = (z>0) * sum_t S2[t,j] dq[s,t]
        for (int i = tid; i < ns * rr; i += nthr) {
            const int s = i / rr, j = i - s * rr;
            float da = 0.0f;
            for (int t = 0; t < T; ++t) da = fmaf(sm[L.se2 + t * rr + j], sm[L.dq + s * T + t], da);
            sm[L.dz + i] = sm[o_z + i] > 0.0f ? da : 0.0f;
        }
    });
    ex.phase([&](int tid) {
        for (int r = tid; r < nr; r += nthr) {   // ds[s,t] = sum_j S1[j,t] dz[s,j]
            const int s = r / T, t = r - s * T;
            float v = 0.0f;
            for (int j = 0; j < rr; ++j) v = fmaf(sm[L.se1 + j * T + t], sm[L.dz + s * rr + j], v);
            sm[o_ds + r] = v;
        }
        for (int i = tid; i < T * rr; i += nthr) {   // parameter gradients, one owner thread per element
            {   // dS2[t,j] += sum_s dq[s,t] relu(z[s,j])      (i = t*rr + j)
                const int t = i / rr, j = i - t * rr;
                float v = 0.0f;
                for (int s = 0; s < ns; ++s) v = fmaf(sm[L.dq + s * T + t], fmaxf(sm[o_z + s * rr + j], 0.0f), v);
                sm[L.a_se2 + i] += v;
            }
            {   // dS1[j,t] += sum_s dz[s,j] pool[s,t]         (i = j*T + t)
                const int j = i / T, t = i - j * T;
                float v = 0.0f;
                for (int s = 0; s < ns; ++s) v = fmaf(sm[L.dz + s * rr + j], sm[o_pool + s * T + t], v);
                sm[L.a_se1 + i] += v;
            }
        }
    });
}

template <int ACT, int TC, int TOKC, int WT>
MMX_D void mlp_block_bwd_body(Exec& ex, const MlpBlockBwdArgs& a) {
    const MlpDims& d = a.d;
    const MlpBlockSmem L = mlp_block_smem(d, true);
    float* sm = ex.smem;
    const int nthr = ex.nthr;
    const int T = d.T, H = d.H, tok = d.tok, ch = d.ch, rr = d.rr, S = d.S, PH = L.PH, PC = L.PC;
    const float* V1 = d.w_in_smem ? sm + L.cw1 : a.w.cw1;
    const float* V2 = d.w_in_smem ? sm + L.cw2 : a.w.cw2;
    const int ldv1 = d.w_in_smem ? PH : H, ldv2 = d.w_in_smem ? PC : ch;
    const Dropout dr = resolve_dropout(a.dr);
    const bool drop = d.training && dr.thresh != 0u;
    const float invH = 1.0f / (float)H;

    // weight-gradient tiling
    const int v1_nt = (H + 3) >> 2, v1_tiles = ((ch + 3) >> 2) * v1_nt;    // dV1 [ch][H]
    const int v2_nt = (ch + 3) >> 2, v2_tiles = ((H + 3) >> 2) * v2_nt;    // dV2 [H][ch]
    const bool persist = v1_tiles <= nthr * WT && v2_tiles <= nthr * WT;
    // token-MLP weight gradients: (output tile, K slice) per thread
    const int w1_nt = (T + 3) >> 2, w1_tiles = ((tok + 3) >> 2) * w1_nt;   // dW1 [tok][T]
    const int w2_nt = (tok + 3) >> 2, w2_tiles = ((T + 3) >> 2) * w2_nt;   // dW2 [T][tok]
    const int tk_tiles = imax(w1_tiles, w2_tiles);
    const int n_slices = imax(1, nthr / tk_tiles);

    PerThread<MlpBwdRegs<WT>> regs(ex);

    ex.phase([&](int tid) {
        mlp_stage_weights(tid, nthr, sm, L, d, a.w);
        zero_vec(tid, nthr, sm + L.a_ln1g, H); zero_vec(tid, nthr, sm + L.a_ln1b, H);
        zero_vec(tid, nthr, sm + L.a_ln2g, H); zero_vec(tid, nthr, sm + L.a_ln2b, H);
        zero_vec(tid, nthr, sm + L.a_cb1, ch); zero_vec(tid, nthr, sm + L.a_cb2, H);
        zero_vec(tid, nthr, sm + L.a_se1, rr * T); zero_vec(tid, nthr, sm + L.a_se2, T * rr);
        zero_vec(tid, nthr, sm + L.a_tb1, tok); zero_vec(tid, nthr, sm + L.a_tb2, T);
        MlpBwdRegs<WT>& rg = regs[tid];
        MMX_UNROLL
        for (int w = 0; w < WT; ++w)
            MMX_UNROLL
            for (int i = 0; i < 4; ++i)
                MMX_UNROLL
                for (int j = 0; j < 4; ++j) { rg.dV1[w][i][j] = 0.0f; rg.dV2[w][i][j] = 0.0f; }
        MMX_UNROLL
        for (int i = 0; i < 4; ++i)
            MMX_UNROLL
            for (int j = 0; j < 4; ++j) { rg.dW1[i][j] = 0.0f; rg.dW2[i][j] = 0.0f; }
    });

    const int ntiles = (d.B + S - 1) / S;
    for (int tile = ex.bid; tile < ntiles; tile += ex.nblk) {
        const long long seq0 = (long long)tile * S;
        const int ns = imin(S, d.B - (int)seq0), nr = ns * T;
        const float* xg = a.x + (size_t)seq0 * T * H;
        const float* dyg = a.dy + (size_t)seq0 * T * H;
        float* dxg = a.dx + (size_t)seq0 * T * H;

        // ---------------- recompute the forward ----------------
        ex.phase([&](int tid) {
            load_tile(tid, nthr, sm + L.bX, xg, nr, H, PH);
            load_tile(tid, nthr, sm + L.bD, dyg, nr, H, PH);
            // zero the WHOLE scratch pad columns once per tile: every buffer below is used as a
            // float4-read GEMM operand at some point, and stale data from the token half of the
            // previous tile may be non-finite
            for (int i = tid; i < nr * (PH - H); i += nthr) {
                const int r = i / (PH - H), c = H + (i - r * (PH - H));
                sm[L.bX1 + r * PH + c] = 0.0f; sm[L.bA + r * PH + c] = 0.0f; sm[L.bY2 + r * PH + c] = 0.0f;
                sm[L.bYt + r * PH + c] = 0.0f;
            }
            for (int i = tid; i < nr * (PC - ch); i += nthr) {
                const int r = i / (PC - ch), c = ch + (i - r * (PC - ch));
                sm[L.bG + r * PC + c] = 0.0f; sm[L.bU + r * PC + c] = 0.0f;
            }
        });
        ln_stats_phases(ex, sm, L.part, L.part2, L.mean1, L.rstd1, sm + L.bX, PH, nr, H);
        ex.phase([&](int tid) {
            TokenMix<ACT, TC, TOKC> tm;
            for (int p = tid; p < ns * H; p += nthr) {
                const int s = p / H, h = p - s * H;
                tm.fwd(sm, L, d, dr, s, h, seq0);
                MMX_UNROLL
                for (int t = 0; t < (TC > 0 ? TC : T); ++t)
                    sm[L.bYt + (s * T + t) * PH + h] = tm.y[t];
            }
        });
        if (d.use_se) {
            row_pool_phases(ex, sm, sm + L.bYt, PH, nr, H, d.use_max, L.pool1, L.amax1, L.part);
            ex.phase([&](int tid) {
                for (int r = tid; r < nr; r += nthr) {
                    const int s = r / T, t = r - s * T;
                    sm[L.gate1 + r] = se_excite(sm + L.se1, sm + L.se2, sm + L.pool1 + s * T, T, rr, t, sm + L.z1 + s * rr);
                }
            });
        }
        ex.phase([&](int tid) {
            for (int i = tid; i < nr * H; i += nthr) {
                const int r = i / H, h = i - r * H;
                const float g = d.use_se ? sm[L.gate1 + r] : 1.0f;
                sm[L.bX1 + r * PH + h] = fmaf(g, sm[L.bYt + r * PH + h], sm[L.bX + r * PH + h]);
            }
        });
        ln_stats_phases(ex, sm, L.part, L.part2, L.mean2, L.rstd2, sm + L.bX1, PH, nr, H);
        ex.phase([&](int tid) {
            for (int i = tid; i < nr * H; i += nthr) {
                const int r = i / H, h = i - r * H;
                sm[L.bA + r * PH + h] = (sm[L.bX1 + r * PH + h] - sm[L.mean2 + r]) * sm[L.rstd2 + r] * sm[L.ln2_g + h] + sm[L.ln2_b + h];
            }
        });
        ex.phase([&](int tid) {
            gemm_nt<4, 4>(tid, nthr, sm + L.bA, PH, V1, ldv1, nr, ch, H, [&](int m, int n, float v) {
                const float u = v + sm[L.cb1 + n];
                sm[L.bU + m * PC + n] = u;
                float gv = act_fwd<ACT>(u);
                if (drop) gv *= dropout_scale(dr, d.site_base + 2, ((unsigned long long)seq0 * T + m) * ch + n);
                sm[L.bG + m * PC + n] = gv;
            });
        });
        ex.phase([&](int tid) {
            gemm_nt<4, 4>(tid, nthr, sm + L.bG, PC, V2, ldv2, nr, H, ch, [&](int m, int n, float v) {
                float yv = v + sm[L.cb2 + n];
                if (drop) yv *= dropout_scale(dr, d.site_base + 3, ((unsigned long long)seq0 * T + m) * H + n);
                sm[L.bY2 + m * PH + n] = yv;
            });
        });
        // ---------------- channel half backward ----------------
        if (d.use_se) {
            row_pool_phases(ex, sm, sm + L.bY2, PH, nr, H, d.use_max, L.pool2, L.amax2, L.part);
            row_dot_phases(ex, sm, sm + L.bD, sm + L.bY2, PH, nr, H, L.dq, L.part2);
            ex.phase([&](int tid) {
                for (int r = tid; r < nr; r += nthr) {
                    const int s = r / T, t = r - s * T;
                    sm[L.gate2 + r] = se_excite(sm + L.se1, sm + L.se2, sm + L.pool2 + s * T, T, rr, t, sm + L.z2 + s * rr);
                }
            });
            se_backward_phases(ex, sm, L, d, ns, L.gate2, L.pool2, L.z2, L.ds2);
        }
        // dY2 = (dOut*gate2 + dpool) * mask2   -> bY2
        ex.phase([&](int tid) {
            for (int i = tid; i < nr * H; i += nthr) {
                const int r = i / H, h = i - r * H;
                float v = sm[L.bD + r * PH + h];
                if (d.use_se) {
                    v *= sm[L.gate2 + r];
                    if (d.use_max) { if ((float)h == sm[L.amax2 + r]) v += sm[L.ds2 + r]; }
                    else v = fmaf(sm[L.ds2 + r], invH, v);
                }
                if (drop) v *= dropout_scale(dr, d.site_base + 3, ((unsigned long long)seq0 * T + r) * H + h);
                sm[L.bY2 + r * PH + h] = v;
            }
        });
        // dc2, dV2 (K = rows) ; dG2 = dY2 V2 ; dU2 = dG2 * mask1 * act'(U2) -> bU (in place)
        ex.phase([&](int tid) {
            for (int h = tid; h < H; h += nthr) {
                float s = 0.0f;
                for (int r = 0; r < nr; ++r) s += sm[L.bY2 + r * PH + h];
                sm[L.a_cb2 + h] += s;
            }
            MlpBwdRegs<WT>& rg = regs[tid];
            if (persist) {
                MMX_UNROLL
                for (int w = 0; w < WT; ++w) {
                    const int t2 = tid + w * nthr;
                    if (t2 < v2_tiles) gemm_tn_acc4x4(rg.dV2[w], t2, v2_nt, sm + L.bY2, PH, sm + L.bG, PC, nr);
                }
            } else {
                for (int t2 = tid; t2 < v2_tiles; t2 += nthr) {
                    float acc[4][4] = {};
                    gemm_tn_acc4x4(acc, t2, v2_nt, sm + L.bY2, PH, sm + L.bG, PC, nr);
                    flush_acc4x4(acc, t2, v2_nt, a.g.cw2, ch, H, ch);
                }
            }
        });
        ex.phase([&](int tid) {
            gemm_nn<4>(tid, nthr, sm + L.bY2, PH, V2, ldv2, nr, ch, H, [&](int m, int n, float v) {
                float ga;
                const float gp = act_fwd_grad<ACT>(sm[L.bU + m * PC + n], &ga);
                if (drop) v *= dropout_scale(dr, d.site_base + 2, ((unsigned long long)seq0 * T + m) * ch + n);
                sm[L.bU + m * PC + n] = v * gp;
            });
        });
        // dc1, dV1 ; dN2 = dU2 V1 -> bY2
        ex.phase([&](int tid) {
            for (int c = tid; c < ch; c += nthr) {
                float s = 0.0f;
                for (int r = 0; r < nr; ++r) s += sm[L.bU + r * PC + c];
                sm[L.a_cb1 + c] += s;
            }
            MlpBwdRegs<WT>& rg = regs[tid];
            if (persist) {
                MMX_UNROLL
                for (int w = 0; w < WT; ++w) {
                    const int t1 = tid + w * nthr;
                    if (t1 < v1_tiles) gemm_tn_acc4x4(rg.dV1[w], t1, v1_nt, sm + L.bU, PC, sm + L.bA, PH, nr);
                }
            } else {
                for (int t1 = tid; t1 < v1_tiles; t1 += nthr) {
                    float acc[4][4] = {};
                    gemm_tn_acc4x4(acc, t1, v1_nt, sm + L.bU, PC, sm + L.bA, PH, nr);
                    flush_acc4x4(acc, t1, v1_nt, a.g.cw1, H, ch, H);
                }
            }
        });
        ex.phase([&](int tid) {
            gemm_nn<4>(tid, nthr, sm + L.bU, PC, V1, ldv1, nr, H, ch, [&](int m, int n, float v) {
                sm[L.bY2 + m * PH + n] = v;
            });
        });
        // LN2 backward: columns -> dgamma2/dbeta2 ; rows -> dX1 = dOut + LN2'(dN2)   (bD in place)
        ex.phase([&](int tid) {
            for (int h = tid; h < H; h += nthr) {
                float sg = 0.0f, sb = 0.0f;
                for (int r = 0; r < nr; ++r) {
                    const float dn = sm[L.bY2 + r * PH + h];
                    const float xh = (sm[L.bX1 + r * PH + h] - sm[L.mean2 + r]) * sm[L.rstd2 + r];
                    sg = fmaf(dn, xh, sg); sb += dn;
                }
                sm[L.a_ln2g + h] += sg; sm[L.a_ln2b + h] += sb;
            }
            for (int i = tid; i < nr * kParts; i += nthr) {       // row partials of m1 = sum dxh, m2 = sum dxh*xhat
                const int r = i / kParts, p = i - r * kParts;
                const float mu = sm[L.mean2 + r], rs = sm[L.rstd2 + r];
                const float* dn = sm + L.bY2 + r * PH;
                const float* x1 = sm + L.bX1 + r * PH;
                float m1 = 0.0f, m2 = 0.0f;
                for (int h = 4 * p; h < H; h += 4 * kParts) {
                    const int n = imin(4, H - h);
                    for (int k = 0; k < n; ++k) {
                        const float dxh = dn[h + k] * sm[L.ln2_g + h + k];
                        m1 += dxh; m2 = fmaf(dxh, (x1[h + k] - mu) * rs, m2);
                    }
                }
                sm[L.part + i] = m1; sm[L.part2 + i] = m2;
            }
        });
        ex.phase([&](int tid) {
            for (int i = tid; i < nr * H; i += nthr) {
                const int r = i / H, h = i - r * H;
                const float mu = sm[L.mean2 + r], rs = sm[L.rstd2 + r];
                const float m1 = sum_parts(sm + L.part + r * kParts) * invH, m2 = sum_parts(sm + L.part2 + r * kParts) * invH;
                const float dxh = sm[L.bY2 + r * PH + h] * sm[L.ln2_g + h];
                sm[L.bD + r * PH + h] += rs * (dxh - m1 - (sm[L.bX1 + r * PH + h] - mu) * rs * m2);
            }
        });
        // ---------------- token half backward ----------------
        if (d.use_se) {
            row_dot_phases(ex, sm, sm + L.bD, sm + L.bYt, PH, nr, H, L.dq, L.part2);
            se_backward_phases(ex, sm, L, d, ns, L.gate1, L.pool1, L.z1, L.ds1);
        }
        ex.phase([&](int tid) {
            // the token-half staging buffers alias the channel-half scratch: clear their pad columns
            for (int i = tid; i < nr * (PH - H); i += nthr) {
                const int r = i / (PH - H), c = H + (i - r * (PH - H));
                sm[L.bN1 + r * PH + c] = 0.0f; sm[L.bdN1 + r * PH + c] = 0.0f;
            }
            for (int i = tid; i < ns * tok * (PH - H); i += nthr) {
                const int r = i / (PH - H), c = H + (i - r * (PH - H));
                sm[L.tG + r * PH + c] = 0.0f; sm[L.tdU + r * PH + c] = 0.0f;
            }
        });
        ex.phase([&](int tid) {
            TokenMix<ACT, TC, TOKC> tm;
            MlpBwdRegs<WT>& rg = regs[tid];
            for (int p = tid; p < ns * H; p += nthr) {
                const int s = p / H, h = p - s * H;
                tm.fwd(sm, L, d, dr, s, h, seq0);
                const unsigned long long pair = (unsigned long long)(seq0 + s) * H + h;
                float dyt[TDim<TC>::cap];
                MMX_UNROLL
                for (int t = 0; t < (TC > 0 ? TC : T); ++t)
                    {
                        const int r = s * T + t;
                        float v = sm[L.bD + r * PH + h];
                        if (d.use_se) {
                            v *= sm[L.gate1 + r];
                            if (d.use_max) { if ((float)h == sm[L.amax1 + r]) v += sm[L.ds1 + r]; }
                            else v = fmaf(sm[L.ds1 + r], invH, v);
                        }
                        if (drop) v *= dropout_scale(dr, d.site_base + 1, pair * T + t);
                        dyt[t] = v;
                        sm[L.bYt + r * PH + h] = v;             // dYt, row-major  (A operand of dW2)
                        sm[L.bN1 + r * PH + h] = tm.n[t];       // N1, row-major   (B operand of dW1)
                    }
                float dn[TDim<TC>::cap];
                MMX_UNROLL
                for (int t = 0; t < (TC > 0 ? TC : T); ++t) dn[t] = 0.0f;
                MMX_UNROLL
                for (int k = 0; k < (TOKC > 0 ? TOKC : tok); ++k)
                    {
                        float dg = 0.0f;
                        MMX_UNROLL
                        for (int t = 0; t < (TC > 0 ? TC : T); ++t)
                            dg = fmaf(sm[L.tw2 + t * tok + k], dyt[t], dg);
                        if (drop) dg *= dropout_scale(dr, d.site_base + 0, pair * tok + k);
                        float ga;
                        const float du = dg * act_fwd_grad<ACT>(tm.u[k], &ga);
                        sm[L.tG + (s * tok + k) * PH + h] = tm.g[k];
                        sm[L.tdU + (s * tok + k) * PH + h] = du;
                        MMX_UNROLL
                        for (int t = 0; t < (TC > 0 ? TC : T); ++t)
                            dn[t] = fmaf(sm[L.tw1 + k * T + t], du, dn[t]);
                    }
                MMX_UNROLL
                for (int t = 0; t < (TC > 0 ? TC : T); ++t)
                    sm[L.bdN1 + (s * T + t) * PH + h] = dn[t];
            }
        });
        // token-MLP weight gradients (split-K over sequences), LN1 backward
        ex.phase([&](int tid) {
            MlpBwdRegs<WT>& rg = regs[tid];
            const int slice = tid / tk_tiles, otile = tid - slice * tk_tiles;
            if (slice < n_slices) {
                const int H4 = (H + 3) >> 2;
                if (otile < w2_tiles) {   // dW2[t][k] += sum_s sum_h dYt[(s,t)][h] G[(s,k)][h]
                    const int mt = otile / w2_nt, nt = otile - mt * w2_nt;
                    for (int s = slice; s < ns; s += n_slices) {
                        const float* A = sm + L.bYt + (s * T) * PH;
                        const float* Bm = sm + L.tG + (s * tok) * PH;
                        for (int q = 0; q < H4; ++q) {
                            f4 av[4], bv[4];
                            MMX_UNROLL
                            for (int i = 0; i < 4; ++i) av[i] = ld4(A + imin(4 * mt + i, T - 1) * PH + 4 * q);
                            MMX_UNROLL
                            for (int j = 0; j < 4; ++j) bv[j] = ld4(Bm + imin(4 * nt + j, tok - 1) * PH + 4 * q);
                            MMX_UNROLL
                            for (int i = 0; i < 4; ++i)
                                MMX_UNROLL
                                for (int j = 0; j < 4; ++j)
                                    rg.dW2[i][j] += (av[i].x * bv[j].x + av[i].y * bv[j].y) + (av[i].z * bv[j].z + av[i].w * bv[j].w);
                        }
                    }
                }
                if (otile < w1_tiles) {   // dW1[k][t] += sum_s sum_h dU[(s,k)][h] N1[(s,t)][h]
                    const int mt = otile / w1_nt, nt = otile - mt * w1_nt;
                    for (int s = slice; s < ns; s += n_slices) {
                        const float* A = sm + L.tdU + (s * tok) * PH;
                        const float* Bm = sm + L.bN1 + (s * T) * PH;
                        for (int q = 0; q < H4; ++q) {
                            f4 av[4], bv[4];
                            MMX_UNROLL
                            for (int i = 0; i < 4; ++i) av[i] = ld4(A + imin(4 * mt + i, tok - 1) * PH + 4 * q);
                            MMX_UNROLL
                            for (int j = 0; j < 4; ++j) bv[j] = ld4(Bm + imin(4 * nt + j, T - 1) * PH + 4 * q);
                            MMX_UNROLL
                            for (int i = 0; i < 4; ++i)
                                MMX_UNROLL
                                for (int j = 0; j < 4; ++j)
                                    rg.dW1[i][j] += (av[i].x * bv[j].x + av[i].y * bv[j].y) + (av[i].z * bv[j].z + av[i].w * bv[j].w);
                        }
                    }
                }
            }
            // token-MLP bias gradients: db1[k] = sum_{s,h} dU[(s,k)][h], db2[t] = sum_{s,h} dYt[(s,t)][h]
            // (8 partial sums per output, combined with shared-memory atomics)
            for (int i = tid; i < (tok + T) * 8; i += nthr) {
                const int o = i >> 3, part = i & 7;
                const bool is1 = o < tok;
                const int rows_per_s = is1 ? tok : T, row_in_s = is1 ? o : o - tok;
                const float* base = sm + (is1 ? L.tdU : L.bYt);
                float sacc = 0.0f;
                for (int s2 = 0; s2 < ns; ++s2) {
                    const float* row = base + (s2 * rows_per_s + row_in_s) * PH;
                    for (int h = part; h < H; h += 8) sacc += row[h];
                }
                smem_add(sm + (is1 ? L.a_tb1 + o : L.a_tb2 + (o - tok)), sacc);
            }
            // LN1 backward, columns: dgamma1/dbeta1
            for (int h = tid; h < H; h += nthr) {
                float sg = 0.0f, sb = 0.0f;
                for (int r = 0; r < nr; ++r) {
                    const float dn = sm[L.bdN1 + r * PH + h];
                    const float xh = (sm[L.bX + r * PH + h] - sm[L.mean1 + r]) * sm[L.rstd1 + r];
                    sg = fmaf(dn, xh, sg); sb += dn;
                }
                sm[L.a_ln1g + h] += sg; sm[L.a_ln1b + h] += sb;
            }
            // LN1 backward, rows: dX = dX1 + LN1'(dN1): row partials of m1, m2 here, the update in the next phase
            for (int i = tid; i < nr * kParts; i += nthr) {
                const int r = i / kParts, p = i - r * kParts;
                const float mu = sm[L.mean1 + r], rs = sm[L.rstd1 + r];
                const float* dn = sm + L.bdN1 + r * PH;
                const float* x0 = sm + L.bX + r * PH;
                float m1 = 0.0f, m2 = 0.0f;
                for (int h = 4 * p; h < H; h += 4 * kParts) {
                    const int n = imin(4, H - h);
                    for (int k = 0; k < n; ++k) {
                        const float dxh = dn[h + k] * sm[L.ln1_g + h + k];
                        m1 += dxh; m2 = fmaf(dxh, (x0[h + k] - mu) * rs, m2);
                    }
                }
                sm[L.part + i] = m1; sm[L.part2 + i] = m2;
            }
        });
        ex.phase([&](int tid) {
            for (int i = tid; i < nr * H; i += nthr) {
                const int r = i / H, h = i - r * H;
                const float mu = sm[L.mean1 + r], rs = sm[L.rstd1 + r];
                const float m1 = sum_parts(sm + L.part + r * kParts) * invH, m2 = sum_parts(sm + L.part2 + r * kParts) * invH;
                const float dxh = sm[L.bdN1 + r * PH + h] * sm[L.ln1_g + h];
                sm[L.bD + r * PH + h] += rs * (dxh - m1 - (sm[L.bX + r * PH + h] - mu) * rs * m2);
            }
        });
        ex.phase([&](int tid) { store_tile(tid, nthr, dxg, sm + L.bD, nr, H, PH); });
    }

    // ---------------- flush the CTA's gradient accumulators ----------------
    ex.phase([&](int tid) { zero_vec(tid, nthr, sm + L.bD, 2 * T * tok); });
    ex.phase([&](int tid) {
        MlpBwdRegs<WT>& rg = regs[tid];
        if (persist) {
            MMX_UNROLL
            for (int w = 0; w < WT; ++w) {
                const int t1 = tid + w * nthr;
                if (t1 < v1_tiles) flush_acc4x4(rg.dV1[w], t1, v1_nt, a.g.cw1, H, ch, H);
                if (t1 < v2_tiles) flush_acc4x4(rg.dV2[w], t1, v2_nt, a.g.cw2, ch, H, ch);
            }
        }
        const int slice = tid / tk_tiles, otile = tid - slice * tk_tiles;
        if (slice < n_slices) {       // combine the CTA's K-split slices in shared memory (tiles bX / bD are idle now)
            if (otile < w2_tiles) smem_add_acc4x4(rg.dW2, otile, w2_nt, sm + L.bD, tok, T, tok);
            if (otile < w1_tiles) smem_add_acc4x4(rg.dW1, otile, w1_nt, sm + L.bD + T * tok, T, tok, T);
        }
        for (int k = tid; k < tok; k += nthr) red_add(a.g.tb1 + k, sm[L.a_tb1 + k]);
        for (int t = tid; t < T; t += nthr) red_add(a.g.tb2 + t, sm[L.a_tb2 + t]);
        for (int h = tid; h < H; h += nthr) {
            red_add(a.g.ln1_g + h, sm[L.a_ln1g + h]); red_add(a.g.ln1_b + h, sm[L.a_ln1b + h]);
            red_add(a.g.ln2_g + h, sm[L.a_ln2g + h]); red_add(a.g.ln2_b + h, sm[L.a_ln2b + h]);
            red_add(a.g.cb2 + h, sm[L.a_cb2 + h]);
        }
        for (int c = tid; c < ch; c += nthr) red_add(a.g.cb1 + c, sm[L.a_cb1 + c]);
        if (d.use_se)
            for (int i = tid; i < T * rr; i += nthr) { red_add(a.g.se1 + i, sm[L.a_se1 + i]); red_add(a.g.se2 + i, sm[L.a_se2 + i]); }
    });
    ex.phase([&](int tid) {
        for (int i = tid; i < T * tok; i += nthr) { red_add(a.g.tw2 + i, sm[L.bD + i]); red_add(a.g.tw1 + i, sm[L.bD + T * tok + i]); }
    });
}


// ------------------------------------------------------------------------------------------
// generic row-tile linear layer:  Y[r][n] = sum_k X[r][k] W[n][k] + b[n]
// Used for the MlpMixer embedding (mlp_mixer.py:325-327: Conv2d(1,H,(1,D)) == per-frame
// Linear(D->H)) and, in mmx_conv.cuh, for the non-harmonic PoseEncoder.embed_mlp.
// ------------------------------------------------------------------------------------------
struct LinearDims { int rows, K, N, R; };   // R = rows per CTA tile
struct LinearSmem { int PK, PN, w, b, x, dy, total; };
MMX_HD LinearSmem linear_smem(const LinearDims& d, bool bwd) {
    LinearSmem L; L.PK = pitch_of(d.K); L.PN = pitch_of(d.N);
    int o = 0;
    L.w = o; o += d.N * L.PK;
    L.b = o; o += round_up(d.N, 4);
    L.x = o; o += d.R * L.PK;
    if (bwd) { L.dy = o; o += d.R * L.PN; } else L.dy = -1;
    L.total = o;
    return L;
}
struct LinearFwdArgs { LinearDims d; const float *x, *w, *b; float* y; };

MMX_D void linear_fwd_body(Exec& ex, const LinearFwdArgs& a) {
    const LinearDims& d = a.d;
    const LinearSmem L = linear_smem(d, false);
    float* sm = ex.smem;
    const int nthr = ex.nthr, K = d.K, N = d.N, R = d.R;
    ex.phase([&](int tid) {
        stage_matrix(tid, nthr, sm + L.w, a.w, N, K, L.PK);
        copy_vec(tid, nthr, sm + L.b, a.b, N);
    });
    const int ntiles = (d.rows + R - 1) / R;
    for (int tile = ex.bid; tile < ntiles; tile += ex.nblk) {
        const int row0 = tile * R, nr = imin(R, d.rows - row0);
        ex.phase([&](int tid) { load_tile(tid, nthr, sm + L.x, a.x + (size_t)row0 * K, nr, K, L.PK); });
        ex.phase([&](int tid) {
            float* yg = a.y + (size_t)row0 * N;
            gemm_nt<4, 4>(tid, nthr, sm + L.x, L.PK, sm + L.w, L.PK, nr, N, K, [&](int m, int n, float v) {
                yg[(size_t)m * N + n] = v + sm[L.b + n];
            });
        });
    }
}

struct LinearBwdArgs { LinearDims d; const float *x, *w, *dy; float *dw, *db, *dx; };  // dx may be null

template <int WT>
struct LinearBwdRegs { float dW[WT][4][4]; };

template <int WT>
MMX_D void linear_bwd_body(Exec& ex, const LinearBwdArgs& a) {
    const LinearDims& d = a.d;
    const LinearSmem L = linear_smem(d, true);
    float* sm = ex.smem;
    const int nthr = ex.nthr, K = d.K, N = d.N, R = d.R;
    const int w_nt = (K + 3) >> 2, w_tiles = ((N + 3) >> 2) * w_nt;   // dW [N][K]
    const bool persist = w_tiles <= nthr * WT;
    PerThread<LinearBwdRegs<WT>> regs(ex);
    float* s_db = sm + L.b;   // bias slot doubles as the db accumulator (the bias itself is not needed)
    ex.phase([&](int tid) {
        if (a.dx) stage_matrix(tid, nthr, sm + L.w, a.w, N, K, L.PK);
        zero_vec(tid, nthr, s_db, N);
        LinearBwdRegs<WT>& rg = regs[tid];
        MMX_UNROLL
        for (int w = 0; w < WT; ++w)
            MMX_UNROLL
            for (int i = 0; i < 4; ++i)
                MMX_UNROLL
                for (int j = 0; j < 4; ++j) rg.dW[w][i][j] = 0.0f;
    });
    const int ntiles = (d.rows + R - 1) / R;
    for (int tile = ex.bid; tile < ntiles; tile += ex.nblk) {
        const int row0 = tile * R, nr = imin(R, d.rows - row0);
        ex.phase([&](int tid) {
            load_tile(tid, nthr, sm + L.x, a.x + (size_t)row0 * K, nr, K, L.PK);
            load_tile(tid, nthr, sm + L.dy, a.dy + (size_t)row0 * N, nr, N, L.PN);
        });
        ex.phase([&](int tid) {
            {
                const int nsl = imax(1, nthr / N);
                for (int it = tid; it < N * nsl; it += nthr) {
                    const int sl = it / N, n = it - sl * N;
                    float s = 0.0f;
                    for (int r = sl; r < nr; r += nsl) s += sm[L.dy + r * L.PN + n];
                    smem_add(s_db + n, s);
                }
            }
            LinearBwdRegs<WT>& rg = regs[tid];
            if (persist) {
                MMX_UNROLL
                for (int w = 0; w < WT; ++w) {
                    const int t = tid + w * nthr;
                    if (t < w_tiles) gemm_tn_acc4x4(rg.dW[w], t, w_nt, sm + L.dy, L.PN, sm + L.x, L.PK, nr);
                }
            } else {
                for (int t = tid; t < w_tiles; t += nthr) {
                    float acc[4][4] = {};
                    gemm_tn_acc4x4(acc, t, w_nt, sm + L.dy, L.PN, sm + L.x, L.PK, nr);
                    flush_acc4x4(acc, t, w_nt, a.dw, K, N, K);
                }
            }
            if (a.dx) {
                float* dxg = a.dx + (size_t)row0 * K;
                gemm_nn<4>(tid, nthr, sm + L.dy, L.PN, sm + L.w, L.PK, nr, K, N, [&](int m, int n, float v) {
                    dxg[(size_t)m * K + n] = v;
                });
            }
        });
    }
    const bool staged = persist && N * K <= R * L.PK;     // dW fits the (now idle) x tile: coalesced flush through shared memory
    ex.phase([&](int tid) {
        LinearBwdRegs<WT>& rg = regs[tid];
        if (persist) {
            MMX_UNROLL
            for (int w = 0; w < WT; ++w) {
                const int t = tid + w * nthr;
                if (t < w_tiles) {
                    if (staged) stage_acc4x4(rg.dW[w], t, w_nt, sm + L.x, K, N, K);
                    else flush_acc4x4(rg.dW[w], t, w_nt, a.dw, K, N, K);
                }
            }
        }
        for (int n = tid; n < N; n += nthr) red_add(a.db + n, s_db[n]);
    });
    if (staged)
        ex.phase([&](int tid) {
            for (int i = tid; i < N * K; i += nthr) red_add(a.dw + i, sm[L.x + i]);
        });
}

// ------------------------------------------------------------------------------------------
// MlpMixer head (mlp_mixer.py:332-335):  Z = LN(X);  P[s,o,:] = sum_t Wt[o,t] Z[s,t,:] + bt[o];
//                                         out[s,o,:] = Wf P[s,o,:] + bf
// ------------------------------------------------------------------------------------------
struct MlpHeadDims { int B, T, To, H, D, S; };
struct MlpHeadW { float *ln_g, *ln_b, *wt, *bt, *wf, *bf; };   // LN.{weight,bias}, conv_out.{weight[To,T,1],bias}, fc_out.{weight[D,H],bias}
struct MlpHeadSmem {
    int PH, PD, ln_g, ln_b, wt, bt, wf, bf, mean, rstd, bX, bP, bO, bZ, a_lng, a_lnb, a_bf, a_bt, a_wt, total;
};
MMX_HD MlpHeadSmem mlp_head_smem(const MlpHeadDims& d, bool bwd) {
    MlpHeadSmem L; L.PH = pitch_of(d.H); L.PD = pitch_of(d.D);
    int o = 0;
    auto take = [&](int n) { int r = o; o += round_up(n, 4); return r; };
    L.ln_g = take(d.H); L.ln_b = take(d.H); L.wt = take(d.To * d.T); L.bt = take(d.To);
    L.wf = take(d.D * L.PH); L.bf = take(d.D);
    L.mean = take(d.S * d.T); L.rstd = take(d.S * d.T);
    L.bX = take(d.S * d.T * L.PH);
    L.bP = take(d.S * d.To * L.PH);
    if (bwd) {
        L.bO = take(d.S * d.To * L.PD);          // dOut tile
        L.bZ = take(d.S * d.T * L.PH);           // Z = LN(X), later dZ
        L.a_lng = take(d.H); L.a_lnb = take(d.H); L.a_bf = take(d.D); L.a_bt = take(d.To); L.a_wt = take(d.To * d.T);
    } else { L.bO = L.bZ = L.a_lng = L.a_lnb = L.a_bf = L.a_bt = L.a_wt = -1; }
    L.total = o;
    return L;
}
struct MlpHeadFwdArgs { MlpHeadDims d; MlpHeadW w; const float* x; float* out; };

template <int TC>
MMX_D void mlp_head_fwd_body(Exec& ex, const MlpHeadFwdArgs& a) {
    const MlpHeadDims& d = a.d;
    const MlpHeadSmem L = mlp_head_smem(d, false);
    float* sm = ex.smem;
    const int nthr = ex.nthr, T = d.T, To = d.To, H = d.H, D = d.D, S = d.S, PH = L.PH;
    ex.phase([&](int tid) {
        copy_vec(tid, nthr, sm + L.ln_g, a.w.ln_g, H); copy_vec(tid, nthr, sm + L.ln_b, a.w.ln_b, H);
        copy_vec(tid, nthr, sm + L.wt, a.w.wt, To * T); copy_vec(tid, nthr, sm + L.bt, a.w.bt, To);
        stage_matrix(tid, nthr, sm + L.wf, a.w.wf, D, H, PH); copy_vec(tid, nthr, sm + L.bf, a.w.bf, D);
    });
    const int ntiles = (d.B + S - 1) / S;
    for (int tile = ex.bid; tile < ntiles; tile += ex.nblk) {
        const long long seq0 = (long long)tile * S;
        const int ns = imin(S, d.B - (int)seq0), nr = ns * T, no = ns * To;
        ex.phase([&](int tid) {
            load_tile(tid, nthr, sm + L.bX, a.x + (size_t)seq0 * T * H, nr, H, PH);
            for (int i = tid; i < no * (PH - H); i += nthr) { const int r = i / (PH - H); sm[L.bP + r * PH + H + (i - r * (PH - H))] = 0.0f; }
        });
        ex.phase([&](int tid) {
            for (int r = tid; r < nr; r += nthr) row_stats(sm + L.bX + r * PH, H, sm + L.mean + r, sm + L.rstd + r, 1e-5f);
        });
        ex.phase([&](int tid) {
            for (int p = tid; p < ns * H; p += nthr) {
                const int s = p / H, h = p - s * H;
                float z[TDim<TC>::cap];
                const float gam = sm[L.ln_g + h], bet = sm[L.ln_b + h];
                MMX_UNROLL
                for (int t = 0; t < (TC > 0 ? TC : T); ++t)
                    { const int r = s * T + t; z[t] = (sm[L.bX + r * PH + h] - sm[L.mean + r]) * sm[L.rstd + r] * gam + bet; }
                for (int o = 0; o < To; ++o) {
                    float acc = sm[L.bt + o];
                    MMX_UNROLL
                    for (int t = 0; t < (TC > 0 ? TC : T); ++t)
                        acc = fmaf(sm[L.wt + o * T + t], z[t], acc);
                    sm[L.bP + (s * To + o) * PH + h] = acc;
                }
            }
        });
        ex.phase([&](int tid) {
            float* og = a.out + (size_t)seq0 * To * D;
            gemm_nt<4, 4>(tid, nthr, sm + L.bP, PH, sm + L.wf, PH, no, D, H, [&](int m, int n, float v) {
                og[(size_t)m * D + n] = v + sm[L.bf + n];
            });
        });
    }
}

struct MlpHeadBwdArgs { MlpHeadDims d; MlpHeadW w; MlpHeadW g; const float* x; const float* dout; float* dx; };

template <int WT>
struct MlpHeadBwdRegs { float dWf[WT][4][4]; float dWt[4][4]; };

template <int TC, int WT>
MMX_D void mlp_head_bwd_body(Exec& ex, const MlpHeadBwdArgs& a) {
    const MlpHeadDims& d = a.d;
    const MlpHeadSmem L = mlp_head_smem(d, true);
    float* sm = ex.smem;
    const int nthr = ex.nthr, T = d.T, To = d.To, H = d.H, D = d.D, S = d.S, PH = L.PH, PD = L.PD;
    const float invH = 1.0f / (float)H;
    const int f_nt = (H + 3) >> 2, f_tiles = ((D + 3) >> 2) * f_nt;        // dWf [D][H]
    const bool persist = f_tiles <= nthr * WT;
    const int t_nt = (T + 3) >> 2, t_tiles = ((To + 3) >> 2) * t_nt;       // dWt [To][T]
    const int n_slices = imax(1, nthr / t_tiles);
    PerThread<MlpHeadBwdRegs<WT>> regs(ex);
    ex.phase([&](int tid) {
        copy_vec(tid, nthr, sm + L.ln_g, a.w.ln_g, H); copy_vec(tid, nthr, sm + L.ln_b, a.w.ln_b, H);
        copy_vec(tid, nthr, sm + L.wt, a.w.wt, To * T); copy_vec(tid, nthr, sm + L.bt, a.w.bt, To);
        stage_matrix(tid, nthr, sm + L.wf, a.w.wf, D, H, PH);
        zero_vec(tid, nthr, sm + L.a_lng, H); zero_vec(tid, nthr, sm + L.a_lnb, H);
        zero_vec(tid, nthr, sm + L.a_bf, D); zero_vec(tid, nthr, sm + L.a_bt, To); zero_vec(tid, nthr, sm + L.a_wt, To * T);
        MlpHeadBwdRegs<WT>& rg = regs[tid];
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
        const int ns = imin(S, d.B - (int)seq0), nr = ns * T, no = ns * To;
        ex.phase([&](int tid) {
            load_tile(tid, nthr, sm + L.bX, a.x + (size_t)seq0 * T * H, nr, H, PH);
            load_tile(tid, nthr, sm + L.bO, a.dout + (size_t)seq0 * To * D, no, D, PD);
            for (int i = tid; i < no * (PH - H); i += nthr) { const int r = i / (PH - H); sm[L.bP + r * PH + H + (i - r * (PH - H))] = 0.0f; }
            for (int i = tid; i < nr * (PH - H); i += nthr) { const int r = i / (PH - H); sm[L.bZ + r * PH + H + (i - r * (PH - H))] = 0.0f; }
        });
        ex.phase([&](int tid) {
            for (int r = tid; r < nr; r += nthr) row_stats(sm + L.bX + r * PH, H, sm + L.mean + r, sm + L.rstd + r, 1e-5f);
        });
        // recompute Z (row-major, kept for dWt) and P
        ex.phase([&](int tid) {
            for (int p = tid; p < ns * H; p += nthr) {
                const int s = p / H, h = p - s * H;
                float z[TDim<TC>::cap];
                const float gam = sm[L.ln_g + h], bet = sm[L.ln_b + h];
                MMX_UNROLL
                for (int t = 0; t < (TC > 0 ? TC : T); ++t)
                    {
                        const int r = s * T + t;
                        z[t] = (sm[L.bX + r * PH + h] - sm[L.mean + r]) * sm[L.rstd + r] * gam + bet;
                        sm[L.bZ + r * PH + h] = z[t];
                    }
                for (int o = 0; o < To; ++o) {
                    float acc = sm[L.bt + o];
                    MMX_UNROLL
                    for (int t = 0; t < (TC > 0 ? TC : T); ++t)
                        acc = fmaf(sm[L.wt + o * T + t], z[t], acc);
                    sm[L.bP + (s * To + o) * PH + h] = acc;
                }
            }
        });
        // dbf, dWf[d][h] += sum_rows dOut[row][d] P[row][h]
        ex.phase([&](int tid) {
            {
                const int nsl = imax(1, nthr / D);            // row slices per column: all threads busy
                for (int it = tid; it < D * nsl; it += nthr) {
                    const int sl = it / D, n = it - sl * D;
                    float s = 0.0f;
                    for (int r = sl; r < no; r += nsl) s += sm[L.bO + r * PD + n];
                    smem_add(sm + L.a_bf + n, s);
                }
            }
            MlpHeadBwdRegs<WT>& rg = regs[tid];
            if (persist) {
                MMX_UNROLL
                for (int w = 0; w < WT; ++w) {
                    const int t = tid + w * nthr;
                    if (t < f_tiles) gemm_tn_acc4x4(rg.dWf[w], t, f_nt, sm + L.bO, PD, sm + L.bP, PH, no);
                }
            } else {
                for (int t = tid; t < f_tiles; t += nthr) {
                    float acc[4][4] = {};
                    gemm_tn_acc4x4(acc, t, f_nt, sm + L.bO, PD, sm + L.bP, PH, no);
                    flush_acc4x4(acc, t, f_nt, a.g.wf, H, D, H);
                }
            }
        });
        // dP = dOut Wf   -> bP (P itself is dead now)
        ex.phase([&](int tid) {
            gemm_nn<4>(tid, nthr, sm + L.bO, PD, sm + L.wf, PH, no, H, D, [&](int m, int n, float v) { sm[L.bP + m * PH + n] = v; });
        });
        // dWt / dbt (split-K over sequences), then dZ per (s,h)
        ex.phase([&](int tid) {
            MlpHeadBwdRegs<WT>& rg = regs[tid];
            const int slice = tid / t_tiles, otile = tid - slice * t_tiles;
            if (slice < n_slices) {
                const int H4 = (H + 3) >> 2;
                const int mt = otile / t_nt, nt = otile - mt * t_nt;
                for (int s = slice; s < ns; s += n_slices) {
                    const float* A = sm + L.bP + (s * To) * PH;
                    const float* Bm = sm + L.bZ + (s * T) * PH;
                    for (int q = 0; q < H4; ++q) {
                        f4 av[4], bv[4];
                        MMX_UNROLL
                        for (int i = 0; i < 4; ++i) av[i] = ld4(A + imin(4 * mt + i, To - 1) * PH + 4 * q);
                        MMX_UNROLL
                        for (int j = 0; j < 4; ++j) bv[j] = ld4(Bm + imin(4 * nt + j, T - 1) * PH + 4 * q);
                        MMX_UNROLL
                        for (int i = 0; i < 4; ++i)
                            MMX_UNROLL
                            for (int j = 0; j < 4; ++j)
                                rg.dWt[i][j] += (av[i].x * bv[j].x + av[i].y * bv[j].y) + (av[i].z * bv[j].z + av[i].w * bv[j].w);
                    }
                }
            }
            for (int i = tid; i < no * 4; i += nthr) {       // dbt[o] = sum_{s,h} dP[(s,o)][h]: (row, quarter) partials
                const int r = i >> 2, part = i & 3;
                const float* row = sm + L.bP + r * PH;
                float s = 0.0f;
                for (int h = 4 * part; h < H; h += 16) {
                    const int n = imin(4, H - h);
                    for (int k = 0; k < n; ++k) s += row[h + k];
                }
                smem_add(sm + L.a_bt + (r % To), s);
            }
        });
        ex.phase([&](int tid) {   // dZ[(s,t)][h] = sum_o Wt[o][t] dP[(s,o)][h]   -> bZ (Z is dead after dWt)
            for (int p = tid; p < ns * H; p += nthr) {
                const int s = p / H, h = p - s * H;
                float dz[TDim<TC>::cap];
                MMX_UNROLL
                for (int t = 0; t < (TC > 0 ? TC : T); ++t) dz[t] = 0.0f;
                for (int o = 0; o < To; ++o) {
                    const float dp = sm[L.bP + (s * To + o) * PH + h];
                    MMX_UNROLL
                    for (int t = 0; t < (TC > 0 ? TC : T); ++t)
                        dz[t] = fmaf(sm[L.wt + o * T + t], dp, dz[t]);
                }
                MMX_UNROLL
                for (int t = 0; t < (TC > 0 ? TC : T); ++t)
                    sm[L.bZ + (s * T + t) * PH + h] = dz[t];
            }
        });
        ex.phase([&](int tid) {   // LN backward: columns (dgamma, dbeta) and rows (dX -> bX in place)
            const int nsl = imax(1, nthr / H);
            for (int it = tid; it < H * nsl; it += nthr) {
                const int sl = it / H, h = it - sl * H;
                float sg = 0.0f, sb = 0.0f;
                for (int r = sl; r < nr; r += nsl) {
                    const float dn = sm[L.bZ + r * PH + h];
                    sg = fmaf(dn, (sm[L.bX + r * PH + h] - sm[L.mean + r]) * sm[L.rstd + r], sg); sb += dn;
                }
                smem_add(sm + L.a_lng + h, sg); smem_add(sm + L.a_lnb + h, sb);
            }
        });
        ex.phase([&](int tid) {
            for (int r = tid; r < nr; r += nthr) {
                const float mu = sm[L.mean + r], rs = sm[L.rstd + r];
                const float* dn = sm + L.bZ + r * PH;
                float* x0 = sm + L.bX + r * PH;
                float m1 = 0.0f, m2 = 0.0f;
                for (int h = 0; h < H; ++h) {
                    const float dxh = dn[h] * sm[L.ln_g + h];
                    m1 += dxh; m2 = fmaf(dxh, (x0[h] - mu) * rs, m2);
                }
                m1 *= invH; m2 *= invH;
                for (int h = 0; h < H; ++h) {
                    const float dxh = dn[h] * sm[L.ln_g + h];
                    x0[h] = rs * (dxh - m1 - (x0[h] - mu) * rs * m2);
                }
            }
        });
        ex.phase([&](int tid) { store_tile(tid, nthr, a.dx + (size_t)seq0 * T * H, sm + L.bX, nr, H, PH); });
    }
    const bool staged = persist && D * H <= S * T * PH;    // dWf fits the (now idle) x tile: coalesced flush through shared memory
    ex.phase([&](int tid) {
        MlpHeadBwdRegs<WT>& rg = regs[tid];
        if (persist) {
            MMX_UNROLL
            for (int w = 0; w < WT; ++w) {
                const int t = tid + w * nthr;
                if (t < f_tiles) {
                    if (staged) stage_acc4x4(rg.dWf[w], t, f_nt, sm + L.bX, H, D, H);
                    else flush_acc4x4(rg.dWf[w], t, f_nt, a.g.wf, H, D, H);
                }
            }
        }
        const int slice = tid / t_tiles, otile = tid - slice * t_tiles;
        if (slice < n_slices) smem_add_acc4x4(rg.dWt, otile, t_nt, sm + L.a_wt, T, To, T);    // combine the CTA's K-split slices
        for (int h = tid; h < H; h += nthr) { red_add(a.g.ln_g + h, sm[L.a_lng + h]); red_add(a.g.ln_b + h, sm[L.a_lnb + h]); }
        for (int n = tid; n < D; n += nthr) red_add(a.g.bf + n, sm[L.a_bf + n]);
        for (int o = tid; o < To; o += nthr) red_add(a.g.bt + o, sm[L.a_bt + o]);
    });
    ex.phase([&](int tid) {
        for (int i = tid; i < To * T; i += nthr) red_add(a.g.wt + i, sm[L.a_wt + i]);
        if (staged)
            for (int i = tid; i < D * H; i += nthr) red_add(a.g.wf + i, sm[L.bX + i]);
    });
}

}  // namespace mmx
