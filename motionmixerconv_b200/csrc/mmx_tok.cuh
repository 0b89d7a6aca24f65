// Token half of a MixerBlock (fp32 CUDA cores, sm_100a), the companion of the tensor-core channel half (mmx_chan_tc5.cuh):
//
//     x1 = x + SE(reg2(fc2(reg1(act(fc1(LN1(x)^T)))))^T)       reference: h36m/mlp_mixer.py:146-155 (MixerBlock.forward, first
//     half), MlpBlock :87-96, SELayer :30-34; restated in oracle/mixer_np.py.
//
// The token MLP contracts over the T frames (K = T and K = tokens_mlp_dim, 10 and 20 in the reference's configurations): far
// too shallow for a tensor-core tile, so it runs as register FMAs, ONE THREAD PER (sequence, hidden column): the thread holds
// its column's T frames in registers as T/2 packed pairs, both contractions are thread-local packed FMAs (fma.rn.f32x2: the
// weight rows come out of shared memory as 64-bit pairs, warp-uniform broadcast reads), and the loop over the hidden units
// j is a rolled loop.  What crosses threads -- LayerNorm statistics, the SE squeeze, the LayerNorm backward sums (all sums
// over the hidden dim of a (sequence, frame) row) -- goes through the shared tile: every thread sums a slice of a row, one
// thread per row adds the slices.  Tiles of S whole sequences enter and leave through the bulk-copy engine
// (cp.async.bulk + mbarrier).
// Backward: forward recomputed; the token weight gradients (a [tok x T] product whose contraction runs over ALL columns of
// ALL sequences) are computed from operands staged in shared memory by "owner" threads with register-resident 4x4 accumulator
// tiles that persist across the CTA's loop over tiles (one flush per CTA).
// Dropout: one keep-bit stream per column covers both sites of the token MLP (bits [0,tok): after the activation, bits
// [tok, tok+T): after fc2) -- tc5::keep8 with row = b*H + h, W8 = ceil((tok+T)/8), site = site_base.
#pragma once
#include "mmx_tc5.cuh"

namespace mmx {
namespace tok {

using namespace tc5;

constexpr int kMaxT = 16;      // frames per sequence served (register arrays)
constexpr int kMaxTok = 32;    // tokens_mlp_dim served (keep bits of one column fit 64 bits together with the T bits)
constexpr int kMaxRRt = 4;
constexpr int kTokThreads = 256;

struct TokArgs {
    const float* x;              // [B,T,H] block input
    const float* dx1;            // backward: gradient wrt x1 (output of the token half) [B,T,H]
    float* out;                  // forward: x1; backward: dx
    float* gate_out;             // forward, nullable: SE gates [B,T] saved for the backward
    const float* x1s;            // backward, nullable: x1 saved by the forward; then `gates` holds its SE gates and the token MLP
    const float* gates;          //   output is recovered as y = (x1 - x) / gate instead of being recomputed
    const float *ln_g, *ln_b, *w1, *b1, *w2, *b2, *se1, *se2;
    float *g_ln_g, *g_ln_b, *g_w1, *g_b1, *g_w2, *g_b2, *g_se1, *g_se2;
    int B, T, H, tok, rr;
    int S;                       // sequences per tile; S*H <= 256, S*T <= 256, T*H % 4 == 0
    int site_base;
    Dropout dr;
    int* abort_count;
};

struct TokSmem {                 // offsets in floats
    int x, d, y, part, stat, sq, gate, w1, w2t, b1, b2, lg, lb, se1, se2, stg, misc, total;
    int cols_pad, rows, PR, TPW;
};
MMX_HD TokSmem tok_smem(int T, int H, int tok, int S, int TT, bool bwd) {
    TokSmem m;
    const int tile = (S * T * H + 3) / 4 * 4 + 4;
    m.rows = S * T;
    m.PR = kTokThreads / m.rows < 1 ? 1 : kTokThreads / m.rows;
    if (m.PR > 8) m.PR = 8;
    m.TPW = (TT + 3) / 4 * 4;
    m.cols_pad = (S * H + 3) / 4 * 4 + 4;
    int o = 0;
    m.x = o; o += tile;
    m.d = o; o += bwd ? tile : 0;
    m.y = o; o += tile;
    m.part = o; o += 2 * m.rows * m.PR;
    m.stat = o; o += 2 * m.rows;            // mean, rstd
    m.sq = o; o += 2 * m.rows;              // squeeze / dgate   (bwd: also m1, m2 of the LayerNorm backward)
    m.gate = o; o += 2 * m.rows;            // gate / ds
    o = (o + 3) / 4 * 4;
    m.w1 = o; o += tok * m.TPW;             // fc1.weight [tok][T] rows, pitch TPW, zero padded
    m.w2t = o; o += tok * m.TPW;            // fc2.weight transposed: [tok][T]
    m.b1 = o; o += (tok + 3) / 4 * 4;
    m.b2 = o; o += m.TPW;
    m.lg = o; o += (H + 3) / 4 * 4;
    m.lb = o; o += (H + 3) / 4 * 4;
    m.se1 = o; o += 32 * kMaxRRt;
    m.se2 = o; o += 32 * kMaxRRt;
    m.stg = o; o += bwd ? (2 * T + 1 + 2 * tok + 1) * m.cols_pad : 0;   // N (T+1 rows: ones last), DYT (T), DU (tok), G (tok+1: ones last)
    m.misc = o; o += 32;                     // barriers, abort flag
    m.total = o;
    return m;
}

MMX_D float2 ffma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }

// excitation of one sequence (T squeeze values at sq[0], sq[stride], ...) for frame t; returns the gate and the pre-activations z
MMX_D float excite(const float* sq, int stride, int t, int T, int rr, const float* se1, const float* se2, float (&z)[kMaxRRt]) {
    float q = 0.0f;
#pragma unroll
    for (int k = 0; k < kMaxRRt; ++k) {
        z[k] = 0.0f;
        if (k < rr) {
            for (int tt = 0; tt < T; ++tt) z[k] = fmaf(se1[k * T + tt], sq[tt * stride], z[k]);
            q = fmaf(se2[t * rr + k], fmaxf(z[k], 0.0f), q);
        }
    }
    return sigmoidf_(q);
}

MMX_D void load_params(float* sm, const TokSmem& m, const TokArgs& a, int tid) {
    const int nt = kTokThreads, T = a.T, tok = a.tok;
    for (int i = tid; i < tok * m.TPW; i += nt) {
        const int j = i / m.TPW, t = i - j * m.TPW;
        sm[m.w1 + i] = t < T ? a.w1[j * T + t] : 0.0f;
        sm[m.w2t + i] = t < T ? a.w2[t * tok + j] : 0.0f;
    }
    for (int i = tid; i < (tok + 3) / 4 * 4; i += nt) sm[m.b1 + i] = i < tok ? a.b1[i] : 0.0f;
    for (int i = tid; i < m.TPW; i += nt) sm[m.b2 + i] = i < T ? a.b2[i] : 0.0f;
    for (int i = tid; i < a.H; i += nt) { sm[m.lg + i] = a.ln_g[i]; sm[m.lb + i] = a.ln_b[i]; }
    for (int i = tid; i < 32 * kMaxRRt; i += nt) {
        sm[m.se1 + i] = (a.rr > 0 && i < a.rr * T) ? a.se1[i] : 0.0f;
        sm[m.se2 + i] = (a.rr > 0 && i < a.rr * T) ? a.se2[i] : 0.0f;
    }
}

// keep bits of one column: bit j (< tok): reg1 element j; bit tok + t: reg2 element t
MMX_D unsigned long long column_keep(const Dropout& dr, uint32_t key, uint32_t colrow, int tok, int T) {
    if (!dr.thresh) return ~0ull;
    const uint32_t n8 = (uint32_t)(tok + T + 7) >> 3;
    unsigned long long k = 0ull;
    for (uint32_t c8 = 0; c8 < n8; ++c8) k |= (unsigned long long)keep8(key, dr.thresh >> 16, colrow, n8, c8) << (8 * c8);
    return k;
}

// weight row j (TT floats, pitch TPW) as TT/2 packed pairs
template <int TT>
MMX_D void load_wrow(const float* p, float2 (&w)[TT / 2]) {
#pragma unroll
    for (int i = 0; i + 1 < TT / 2; i += 2) {
        const float4 v = *reinterpret_cast<const float4*>(p + 2 * i);
        w[i] = make_float2(v.x, v.y);
        w[i + 1] = make_float2(v.z, v.w);
    }
    if ((TT / 2) & 1) w[TT / 2 - 1] = *reinterpret_cast<const float2*>(p + TT - 2);
}

// forward of one column: n (normalised, affine) -> y (token MLP output after reg2), packed pairs over t
template <int ACT, int TT>
MMX_D void column_fwd(const float* sm, const TokSmem& m, int tok, const float2 (&n)[TT / 2], float2 (&y)[TT / 2], unsigned long long keep,
                      float scale) {
#pragma unroll
    for (int p = 0; p < TT / 2; ++p) y[p] = *reinterpret_cast<const float2*>(sm + m.b2 + 2 * p);
#pragma unroll 2
    for (int j = 0; j < tok; ++j) {
        float2 w[TT / 2];
        load_wrow<TT>(sm + m.w1 + j * m.TPW, w);
        float2 acc = make_float2(sm[m.b1 + j], 0.0f);
#pragma unroll
        for (int p = 0; p < TT / 2; ++p) acc = ffma2(w[p], n[p], acc);
        float gv = act_fwd<ACT>(acc.x + acc.y);
        gv = (keep >> j) & 1ull ? gv * scale : 0.0f;
        load_wrow<TT>(sm + m.w2t + j * m.TPW, w);
        const float2 gg = make_float2(gv, gv);
#pragma unroll
        for (int p = 0; p < TT / 2; ++p) y[p] = ffma2(w[p], gg, y[p]);
    }
#pragma unroll
    for (int p = 0; p < TT / 2; ++p) {
        y[p].x = (keep >> (tok + 2 * p)) & 1ull ? y[p].x * scale : 0.0f;
        y[p].y = (keep >> (tok + 2 * p + 1)) & 1ull ? y[p].y * scale : 0.0f;
    }
}

// partial sums of every row of a dense [rows][H] tile by all threads: thread -> (row, slice); f(row, h) returns the two
// addends.  Results land in part[(row * PR + slice) * 2 + {0,1}]; combine with row_total() after a CTA barrier.
template <class F>
MMX_D void row_partials(float* sm, const TokSmem& m, int nrows, int H, int tid, F&& f) {
    const int row = tid / m.PR, sl = tid - row * m.PR;
    if (row < nrows) {
        float a = 0.0f, b = 0.0f;
        for (int h = 2 * sl; h < H; h += 2 * m.PR) {      // H is even: column pairs, 64-bit shared loads
            float u, v;
            f(row, h, u, v);
            a += u;
            b += v;
        }
        sm[m.part + (row * m.PR + sl) * 2] = a;
        sm[m.part + (row * m.PR + sl) * 2 + 1] = b;
    }
}
MMX_D void row_total(const float* sm, const TokSmem& m, int row, float& a, float& b) {
    a = 0.0f; b = 0.0f;
    for (int s = 0; s < m.PR; ++s) { a += sm[m.part + (row * m.PR + s) * 2]; b += sm[m.part + (row * m.PR + s) * 2 + 1]; }
}

// LayerNorm statistics of the x tile (shifted one-pass: the shift is the row's first element).  Two CTA barriers.
MMX_D void ln_stats(float* sm, const TokSmem& m, int nrows, int H, int tid) {
    row_partials(sm, m, nrows, H, tid, [&](int r, int h, float& u, float& v) {
        const float2 xv = *reinterpret_cast<const float2*>(sm + m.x + r * H + h);
        const float c0 = sm[m.x + r * H], d0 = xv.x - c0, d1 = xv.y - c0;
        u = d0 + d1; v = fmaf(d0, d0, d1 * d1);
    });
    __syncthreads();
    if (tid < nrows) {
        float s, ss;
        row_total(sm, m, tid, s, ss);
        const float ms = s / (float)H;
        sm[m.stat + 2 * tid] = sm[m.x + tid * H] + ms;
        sm[m.stat + 2 * tid + 1] = 1.0f / sqrtf(fmaxf(ss / (float)H - ms * ms, 0.0f) + 1e-5f);
    }
    __syncthreads();
}

// ==========================================================================================
// forward:  x -> x1
// ==========================================================================================
template <int ACT, int TT>
__global__ void __launch_bounds__(kTokThreads) tok_fwd_kernel(const TokArgs a) {
    constexpr bool EX = TT == 10;      // this instantiation is dispatched for T == 10 only: no t < T predicates
    extern __shared__ float4 tok_smem_raw[];
    float* sm = reinterpret_cast<float*>(tok_smem_raw);
    const TokSmem m = tok_smem(a.T, a.H, a.tok, a.S, TT, false);
    uint64_t* bars = reinterpret_cast<uint64_t*>(sm + m.misc);
    volatile int* abortf = reinterpret_cast<volatile int*>(sm + m.misc + 8);
    const int tid = threadIdx.x, T = a.T, H = a.H, S = a.S, rr = a.rr, tok = a.tok;
    const Dropout dr = resolve_dropout(a.dr);
    const uint32_t key = drop_key(dr.seed_lo, dr.seed_hi, a.site_base, dr.step);
    if (tid == 0) { mbar_init(&bars[0], 1); *abortf = 0; fence_mbar_init(); }
    pdl_launch_dependents();
    load_params(sm, m, a, tid);        // parameters only: overlaps the previous kernel's tail
    __syncthreads();
    pdl_wait();                        // the previous kernel has completed: x is readable
    const int ntiles = (a.B + S - 1) / S;
    const int s_l = tid / H, h = tid - s_l * H;
    const bool col_ok = tid < S * H;
    uint32_t ph = 0;
    auto tile_bytes = [&](int tile) { return (uint32_t)(min(S, a.B - tile * S) * T * H) * 4u; };
    if (tid == 0 && (int)blockIdx.x < ntiles) {
        mbar_expect_tx(&bars[0], tile_bytes(blockIdx.x));
        bulk_g2s(sm + m.x, a.x + (size_t)blockIdx.x * S * T * H, tile_bytes(blockIdx.x), &bars[0]);
    }
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int nseq = min(S, a.B - tile * S);
        const int nrows = nseq * T;
        mbar_wait(&bars[0], ph, abortf);
        ph ^= 1;
        ln_stats(sm, m, nrows, H, tid);
        // ---- token MLP of the thread's column
        const bool act_col = col_ok && s_l < nseq;
        float2 x[TT / 2], y[TT / 2];
        if (act_col) {
            float2 n[TT / 2];
            const float gmm = sm[m.lg + h], bta = sm[m.lb + h];
#pragma unroll
            for (int t = 0; t < TT; ++t) {
                float xv = 0.0f, nv = 0.0f;
                if (EX || t < T) {
                    const int r = s_l * T + t;
                    xv = sm[m.x + r * H + h];
                    const float2 st = *reinterpret_cast<const float2*>(sm + m.stat + 2 * r);
                    nv = fmaf((xv - st.x) * st.y, gmm, bta);
                }
                if (t & 1) { x[t / 2].y = xv; n[t / 2].y = nv; } else { x[t / 2].x = xv; n[t / 2].x = nv; }
            }
            const unsigned long long keep = column_keep(dr, key, (uint32_t)((size_t)(tile * S + s_l) * H + h), tok, T);
            column_fwd<ACT, TT>(sm, m, tok, n, y, keep, dr.scale);
            if (rr > 0) {
#pragma unroll
                for (int t = 0; t < TT; ++t)
                    if (EX || t < T) sm[m.y + (s_l * T + t) * H + h] = (t & 1) ? y[t / 2].y : y[t / 2].x;
            }
        }
        if (rr > 0) {
            __syncthreads();
            // ---- squeeze (mean over the hidden dim of every row) and excitation
            row_partials(sm, m, nrows, H, tid, [&](int r, int hh, float& u, float& v) {
                const float2 yv = *reinterpret_cast<const float2*>(sm + m.y + r * H + hh);
                u = yv.x + yv.y; v = 0.0f;
            });
            __syncthreads();
            if (tid < nrows) {
                float s, dummy;
                row_total(sm, m, tid, s, dummy);
                sm[m.sq + 2 * tid] = s / (float)H;
            }
            __syncthreads();
            if (tid < nrows) {
                float z[kMaxRRt];
                const int sq0 = (tid / T) * T;
                const float gte = excite(sm + m.sq + 2 * sq0, 2, tid - sq0, T, rr, sm + m.se1, sm + m.se2, z);
                sm[m.gate + 2 * tid] = gte;
                if (a.gate_out) a.gate_out[(size_t)tile * S * T + tid] = gte;
            }
            __syncthreads();
        }
        // ---- gate + residual, in place in the x tile
        if (act_col) {
#pragma unroll
            for (int t = 0; t < TT; ++t)
                if (EX || t < T) {
                    const int r = s_l * T + t;
                    const float gte = rr > 0 ? sm[m.gate + 2 * r] : 1.0f;
                    const float yv = (t & 1) ? y[t / 2].y : y[t / 2].x, xv = (t & 1) ? x[t / 2].y : x[t / 2].x;
                    sm[m.x + r * H + h] = fmaf(yv, gte, xv);
                }
        }
        fence_async_smem();
        __syncthreads();
        if (tid == 0) {
            bulk_s2g(a.out + (size_t)tile * S * T * H, sm + m.x, (uint32_t)nrows * H * 4u);
            bulk_commit();
            const int next = tile + gridDim.x;
            bulk_wait_read0();                 // the x tile is both the store source and the next load's destination
            if (next < ntiles) {
                mbar_expect_tx(&bars[0], tile_bytes(next));
                bulk_g2s(sm + m.x, a.x + (size_t)next * S * T * H, tile_bytes(next), &bars[0]);
            }
        }
    }
    if (tid == 0) {
        bulk_wait_all0();
        if (*abortf) atomicAdd(a.abort_count, 1);
    }
}

// ==========================================================================================
// backward:  (x, dx1) -> dx, parameter gradients of the token half
// ==========================================================================================
template <int ACT, int TT>
__global__ void __launch_bounds__(kTokThreads, 2) tok_bwd_kernel(const TokArgs a) {
    constexpr bool EX = TT == 10;
    extern __shared__ float4 tok_smem_raw[];
    float* sm = reinterpret_cast<float*>(tok_smem_raw);
    const TokSmem m = tok_smem(a.T, a.H, a.tok, a.S, TT, true);
    uint64_t* bars = reinterpret_cast<uint64_t*>(sm + m.misc);
    volatile int* abortf = reinterpret_cast<volatile int*>(sm + m.misc + 8);
    constexpr int NT = kTokThreads;
    const int tid = threadIdx.x, T = a.T, H = a.H, S = a.S, rr = a.rr, tok = a.tok;
    const Dropout dr = resolve_dropout(a.dr);
    const uint32_t key = drop_key(dr.seed_lo, dr.seed_hi, a.site_base, dr.step);
    if (tid == 0) { mbar_init(&bars[0], 1); *abortf = 0; fence_mbar_init(); }
    pdl_launch_dependents();
    load_params(sm, m, a, tid);        // parameters only: overlaps the previous kernel's tail
    // staging area: rows [0,T] = N (row T: ones), [T+1, 2T] = DYT, [2T+1, 2T+tok] = DU, [2T+tok+1, 2T+2tok+1] = G (last: ones)
    const int CP = m.cols_pad;
    float* sN = sm + m.stg;
    float* sDYT = sN + (T + 1) * CP;
    float* sDU = sDYT + T * CP;
    float* sG = sDU + tok * CP;
    for (int i = tid; i < (2 * T + 2 * tok + 2) * CP; i += NT) sm[m.stg + i] = 0.0f;
    __syncthreads();
    for (int i = tid; i < S * H; i += NT) { sN[T * CP + i] = 1.0f; sG[tok * CP + i] = 1.0f; }
    __syncthreads();

    const int ntiles = (a.B + S - 1) / S;
    const int s_l = tid / H, h = tid - s_l * H;
    const bool col_ok = tid < S * H;
    // ---- owner threads of the weight-gradient tiles
    //   product 0: dW1ext[j][t'] = sum_col DU[j][col] * N[t'][col]       (j < tok, t' <= T; column T = db1)
    //   product 1: dW2ext[t][j'] = sum_col DYT[t][col] * G[j'][col]      (t < T, j' <= tok; column tok = db2)
    const int nb0r = (tok + 3) / 4, nb0c = (T + 1 + 3) / 4, nb1r = (T + 3) / 4, nb1c = (tok + 1 + 3) / 4;
    const int nblocks = nb0r * nb0c + nb1r * nb1c;
    const int KS = max(1, NT / nblocks);
    const int ob = tid / KS, oks = tid - ob * KS;
    const bool owner = ob < nblocks;
    const int oprod = ob < nb0r * nb0c ? 0 : 1;
    const int obb = oprod ? ob - nb0r * nb0c : ob;
    const int obr = oprod ? obb / nb1c : obb / nb0c, obc = oprod ? obb - obr * nb1c : obb - obr * nb0c;
    const float* oA = oprod ? sDYT : sDU;
    const float* oB = oprod ? sG : sN;
    const int oAr = oprod ? T : tok, oBr = oprod ? tok + 1 : T + 1;
    float2 acc[4][4];     // packed partial sums over even / odd columns
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = make_float2(0.0f, 0.0f);
    float g_lg = 0.0f, g_lb = 0.0f;                  // dLN1.weight[h], dLN1.bias[h] of the thread's column
    float gS1[kMaxRRt], gS2[kMaxRRt];
#pragma unroll
    for (int k = 0; k < kMaxRRt; ++k) gS1[k] = gS2[k] = 0.0f;

    uint32_t ph = 0;
    auto tile_bytes = [&](int tile) { return (uint32_t)(min(S, a.B - tile * S) * T * H) * 4u; };
    pdl_wait();                        // the previous kernel (the channel half backward) has completed: dx1 is readable
    const bool saved = a.x1s != nullptr && rr > 0;      // y recovered from the saved x1 (needed for the SE backward only)
    if (tid == 0 && (int)blockIdx.x < ntiles) {
        mbar_expect_tx(&bars[0], (saved ? 3 : 2) * tile_bytes(blockIdx.x));
        bulk_g2s(sm + m.x, a.x + (size_t)blockIdx.x * S * T * H, tile_bytes(blockIdx.x), &bars[0]);
        bulk_g2s(sm + m.d, a.dx1 + (size_t)blockIdx.x * S * T * H, tile_bytes(blockIdx.x), &bars[0]);
        if (saved) bulk_g2s(sm + m.y, a.x1s + (size_t)blockIdx.x * S * T * H, tile_bytes(blockIdx.x), &bars[0]);
    }
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int nseq = min(S, a.B - tile * S);
        const int nrows = nseq * T;
        mbar_wait(&bars[0], ph, abortf);
        ph ^= 1;
        if (saved && tid < nrows) {                     // 1 / gate of every row (read by the squeeze pass below)
            const float gte = a.gates[(size_t)tile * S * T + tid];
            sm[m.sq + 2 * tid + 1] = gte > 1e-30f ? 1.0f / gte : 0.0f;
        }
        ln_stats(sm, m, nrows, H, tid);
        // ---- forward of the column (n, y)
        const bool act_col = col_ok && s_l < nseq;
        const unsigned long long keep = act_col ? column_keep(dr, key, (uint32_t)((size_t)(tile * S + s_l) * H + h), tok, T) : 0ull;
        float2 n[TT / 2], xh[TT / 2], dyt[TT / 2];
        const float gmm = col_ok ? sm[m.lg + h] : 0.0f, bta = col_ok ? sm[m.lb + h] : 0.0f;
        if (act_col) {
#pragma unroll
            for (int t = 0; t < TT; ++t) {
                float xv = 0.0f, nv = 0.0f;
                if (EX || t < T) {
                    const int r = s_l * T + t;
                    const float2 st = *reinterpret_cast<const float2*>(sm + m.stat + 2 * r);
                    xv = (sm[m.x + r * H + h] - st.x) * st.y;
                    nv = fmaf(xv, gmm, bta);
                }
                if (t & 1) { xh[t / 2].y = xv; n[t / 2].y = nv; } else { xh[t / 2].x = xv; n[t / 2].x = nv; }
            }
            if (rr > 0 && !saved) {
                float2 y[TT / 2];
                column_fwd<ACT, TT>(sm, m, tok, n, y, keep, dr.scale);
#pragma unroll
                for (int t = 0; t < TT; ++t)
                    if (EX || t < T) sm[m.y + (s_l * T + t) * H + h] = (t & 1) ? y[t / 2].y : y[t / 2].x;
            }
        }
        if (rr > 0) {
            __syncthreads();
            // ---- squeeze and d(gate) per row
            row_partials(sm, m, nrows, H, tid, [&](int r, int hh, float& u, float& v) {
                float2 yv = *reinterpret_cast<const float2*>(sm + m.y + r * H + hh);
                const float2 dv = *reinterpret_cast<const float2*>(sm + m.d + r * H + hh);
                if (saved) {                            // the y tile holds x1:  y = (x1 - x) / gate
                    const float2 xv = *reinterpret_cast<const float2*>(sm + m.x + r * H + hh);
                    const float ig = sm[m.sq + 2 * r + 1];
                    yv.x = (yv.x - xv.x) * ig; yv.y = (yv.y - xv.y) * ig;
                }
                u = yv.x + yv.y; v = fmaf(yv.x, dv.x, yv.y * dv.y);
            });
            __syncthreads();
            if (tid < nrows) {
                float s, dg;
                row_total(sm, m, tid, s, dg);
                sm[m.sq + 2 * tid] = s / (float)H;
                sm[m.sq + 2 * tid + 1] = dg;
            }
            __syncthreads();
            // ---- excitation forward + backward of the row's sequence
            if (tid < nrows) {
                const int sq0 = (tid / T) * T, t = tid - sq0;
                float z[kMaxRRt];
                const float gate = excite(sm + m.sq + 2 * sq0, 2, t, T, rr, sm + m.se1, sm + m.se2, z);
                float da[kMaxRRt];
#pragma unroll
                for (int k = 0; k < kMaxRRt; ++k) da[k] = 0.0f;
                float dq_own = 0.0f;
                for (int tt = 0; tt < T; ++tt) {
                    float q = 0.0f;
#pragma unroll
                    for (int k = 0; k < kMaxRRt; ++k)
                        if (k < rr) q = fmaf(sm[m.se2 + tt * rr + k], fmaxf(z[k], 0.0f), q);
                    const float gt = sigmoidf_(q);
                    const float dq = sm[m.sq + 2 * (sq0 + tt) + 1] * gt * (1.0f - gt);
                    if (tt == t) dq_own = dq;
#pragma unroll
                    for (int k = 0; k < kMaxRRt; ++k)
                        if (k < rr) da[k] = fmaf(dq, sm[m.se2 + tt * rr + k], da[k]);
                }
                float ds = 0.0f;
#pragma unroll
                for (int k = 0; k < kMaxRRt; ++k)
                    if (k < rr) {
                        const float dz = z[k] > 0.0f ? da[k] : 0.0f;
                        ds = fmaf(dz, sm[m.se1 + k * T + t], ds);
                        gS2[k] = fmaf(dq_own, fmaxf(z[k], 0.0f), gS2[k]);
                        gS1[k] = fmaf(dz, sm[m.sq + 2 * tid], gS1[k]);
                    }
                sm[m.gate + 2 * tid] = gate;
                sm[m.gate + 2 * tid + 1] = ds / (float)H;
            }
            __syncthreads();
        }
        // ---- backward of the column
        float2 dnh[TT / 2];
        if (act_col) {
#pragma unroll
            for (int t = 0; t < TT; ++t) {
                float v = 0.0f;
                if (EX || t < T) {
                    const int r = s_l * T + t;
                    const float d1 = sm[m.d + r * H + h];
                    const float2 gd = *reinterpret_cast<const float2*>(sm + m.gate + 2 * r);
                    v = rr > 0 ? fmaf(d1, gd.x, gd.y) : d1;
                    v = (keep >> (tok + t)) & 1ull ? v * dr.scale : 0.0f;
                    sDYT[t * CP + tid] = v;
                }
                if (t & 1) dyt[t / 2].y = v; else dyt[t / 2].x = v;
            }
            float2 dn[TT / 2];
#pragma unroll
            for (int p = 0; p < TT / 2; ++p) dn[p] = make_float2(0.0f, 0.0f);
#pragma unroll 2
            for (int j = 0; j < tok; ++j) {
                float2 w1r[TT / 2], w2r[TT / 2];
                load_wrow<TT>(sm + m.w1 + j * m.TPW, w1r);
                load_wrow<TT>(sm + m.w2t + j * m.TPW, w2r);
                float2 au = make_float2(sm[m.b1 + j], 0.0f), ag = make_float2(0.0f, 0.0f);
#pragma unroll
                for (int p = 0; p < TT / 2; ++p) { au = ffma2(w1r[p], n[p], au); ag = ffma2(w2r[p], dyt[p], ag); }
                float av;
                const float dact = act_fwd_grad<ACT>(au.x + au.y, &av);
                const float ksc = (keep >> j) & 1ull ? dr.scale : 0.0f;
                const float du = (ag.x + ag.y) * dact * ksc;
                const float2 dd = make_float2(du, du);
#pragma unroll
                for (int p = 0; p < TT / 2; ++p) dn[p] = ffma2(w1r[p], dd, dn[p]);
                sDU[j * CP + tid] = du;
                sG[j * CP + tid] = av * ksc;
            }
#pragma unroll
            for (int t = 0; t < TT; ++t)
                if (EX || t < T) {
                    const float nv = (t & 1) ? n[t / 2].y : n[t / 2].x, dv = (t & 1) ? dn[t / 2].y : dn[t / 2].x;
                    const float xv = (t & 1) ? xh[t / 2].y : xh[t / 2].x;
                    sN[t * CP + tid] = nv;
                    g_lg = fmaf(dv, xv, g_lg);
                    g_lb += dv;
                    const float dh = dv * gmm;
                    if (t & 1) dnh[t / 2].y = dh; else dnh[t / 2].x = dh;
                    sm[m.y + (s_l * T + t) * H + h] = dh;
                }
        } else if (col_ok) {
            for (int j = 0; j < tok; ++j) { sDU[j * CP + tid] = 0.0f; sG[j * CP + tid] = 0.0f; }
            for (int t = 0; t < T; ++t) { sN[t * CP + tid] = 0.0f; sDYT[t * CP + tid] = 0.0f; }
        }
        __syncthreads();
        // ---- LayerNorm backward row sums; weight-gradient tiles
        row_partials(sm, m, nrows, H, tid, [&](int r, int hh, float& u, float& v) {
            const float2 dv = *reinterpret_cast<const float2*>(sm + m.y + r * H + hh);
            const float2 xv = *reinterpret_cast<const float2*>(sm + m.x + r * H + hh);
            const float2 st = *reinterpret_cast<const float2*>(sm + m.stat + 2 * r);
            u = dv.x + dv.y; v = fmaf(dv.x, (xv.x - st.x) * st.y, dv.y * ((xv.y - st.x) * st.y));
        });
        if (owner) {
            const float* ar[4];
            const float* br[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                ar[i] = oA + (size_t)min(4 * obr + i, oAr - 1) * CP;
                br[i] = oB + (size_t)min(4 * obc + i, oBr - 1) * CP;
            }
#pragma unroll 1
            for (int q = oks; q < CP / 4; q += KS) {
                float4 av[4], bv[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) { av[i] = *reinterpret_cast<const float4*>(ar[i] + 4 * q); bv[i] = *reinterpret_cast<const float4*>(br[i] + 4 * q); }
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        acc[i][j] = ffma2(make_float2(av[i].x, av[i].y), make_float2(bv[j].x, bv[j].y), acc[i][j]);
                        acc[i][j] = ffma2(make_float2(av[i].z, av[i].w), make_float2(bv[j].z, bv[j].w), acc[i][j]);
                    }
            }
        }
        __syncthreads();
        if (tid < nrows) {
            float s1, s2;
            row_total(sm, m, tid, s1, s2);
            sm[m.sq + 2 * tid] = s1 / (float)H;
            sm[m.sq + 2 * tid + 1] = s2 / (float)H;
        }
        __syncthreads();
        // ---- dx = dx1 + LN1 backward, in place in the dx1 tile
        if (act_col) {
#pragma unroll
            for (int t = 0; t < TT; ++t)
                if (EX || t < T) {
                    const int r = s_l * T + t;
                    const float rstd = sm[m.stat + 2 * r + 1];
                    const float2 mm = *reinterpret_cast<const float2*>(sm + m.sq + 2 * r);
                    const float dh = (t & 1) ? dnh[t / 2].y : dnh[t / 2].x, xv = (t & 1) ? xh[t / 2].y : xh[t / 2].x;
                    sm[m.d + r * H + h] += rstd * (dh - mm.x - xv * mm.y);
                }
        }
        fence_async_smem();
        __syncthreads();
        if (tid == 0) {
            bulk_s2g(a.out + (size_t)tile * S * T * H, sm + m.d, (uint32_t)nrows * H * 4u);
            bulk_commit();
            const int next = tile + gridDim.x;
            bulk_wait_read0();
            if (next < ntiles) {
                mbar_expect_tx(&bars[0], (saved ? 3 : 2) * tile_bytes(next));
                bulk_g2s(sm + m.x, a.x + (size_t)next * S * T * H, tile_bytes(next), &bars[0]);
                bulk_g2s(sm + m.d, a.dx1 + (size_t)next * S * T * H, tile_bytes(next), &bars[0]);
                if (saved) bulk_g2s(sm + m.y, a.x1s + (size_t)next * S * T * H, tile_bytes(next), &bars[0]);
            }
        }
    }
    if (tid == 0) bulk_wait_all0();
    __syncthreads();
    // ---------------- flush
    float* red = sm + m.stg;           // staging area is free now
    const int n0 = tok * (T + 1), n1 = T * (tok + 1);
    for (int i = tid; i < n0 + n1 + 2 * H + 2 * 32 * kMaxRRt; i += NT) red[i] = 0.0f;
    __syncthreads();
    // owner tiles: [block][kslice][16] partial sums -> summed over the K slices by one thread per output element
    float* own = red + n0 + n1 + 2 * H + 2 * 32 * kMaxRRt;
    if (owner) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) own[(ob * KS + oks) * 16 + i * 4 + j] = acc[i][j].x + acc[i][j].y;
    }
    __syncthreads();
    for (int e = tid; e < nblocks * 16; e += NT) {
        const int b = e >> 4, i = (e >> 2) & 3, j = e & 3;
        float v = 0.0f;
        for (int ks = 0; ks < KS; ++ks) v += own[(b * KS + ks) * 16 + i * 4 + j];
        const int prod = b < nb0r * nb0c ? 0 : 1, bb = prod ? b - nb0r * nb0c : b;
        const int br_ = prod ? bb / nb1c : bb / nb0c, bc_ = prod ? bb - br_ * nb1c : bb - br_ * nb0c;
        const int r = 4 * br_ + i, c = 4 * bc_ + j;
        if (prod == 0) { if (r < tok && c <= T) red[r * (T + 1) + c] = v; }
        else { if (r < T && c <= tok) red[n0 + r * (tok + 1) + c] = v; }
    }
    if (col_ok) {
        atomicAdd(red + n0 + n1 + h, g_lg);
        atomicAdd(red + n0 + n1 + H + h, g_lb);
    }
    if (rr > 0 && tid < S * T) {
        const int t = tid % T;
        float* rs = red + n0 + n1 + 2 * H;
        for (int k = 0; k < rr; ++k) {
            atomicAdd(rs + k * T + t, gS1[k]);
            atomicAdd(rs + 32 * kMaxRRt + t * rr + k, gS2[k]);
        }
    }
    __syncthreads();
    for (int i = tid; i < tok * T; i += NT) {
        const int j = i / T, t = i - j * T;
        red_add(a.g_w1 + i, red[j * (T + 1) + t]);
        const int t2 = i / tok, j2 = i - t2 * tok;
        red_add(a.g_w2 + i, red[n0 + t2 * (tok + 1) + j2]);
    }
    for (int j = tid; j < tok; j += NT) red_add(a.g_b1 + j, red[j * (T + 1) + T]);
    for (int t = tid; t < T; t += NT) red_add(a.g_b2 + t, red[n0 + t * (tok + 1) + tok]);
    for (int i = tid; i < H; i += NT) { red_add(a.g_ln_g + i, red[n0 + n1 + i]); red_add(a.g_ln_b + i, red[n0 + n1 + H + i]); }
    if (rr > 0)
        for (int i = tid; i < rr * T; i += NT) {
            red_add(a.g_se1 + i, red[n0 + n1 + 2 * H + i]);
            red_add(a.g_se2 + i, red[n0 + n1 + 2 * H + 32 * kMaxRRt + i]);
        }
    if (tid == 0 && *abortf) atomicAdd(a.abort_count, 1);
}

}  // namespace tok
}  // namespace mmx
