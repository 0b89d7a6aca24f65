// MixerBlock forward / backward, warp-per-sequence-pair variant (hidden_dim, channels_mlp_dim <= 64).
//
// Reference arithmetic: h36m/mlp_mixer.py:138-164 (same as mmx_mlp.cuh, which stays the generic variant).
//
// Every warp owns TWO sequences at a time (16 lanes each); lane q of a sequence owns hidden columns
// 4q..4q+3 of all T frames in registers.  Nothing in the main loop needs a CTA barrier: LayerNorm / SE row
// reductions go through a per-warp shared-memory exchange, the token-mixing MLP runs entirely in the
// lane's registers (contraction over T / tokens_mlp_dim), the channel-mixing contractions are warp-level
// register-tiled GEMMs whose A operand is the warp's own [T x H] tile in shared memory and whose B operand
// is the CTA-shared weight matrix.  Backward: the forward is recomputed; dV1 / dV2 are accumulated per
// sequence pair by a warp-level outer-product GEMM into XOR-swizzled (bank-conflict-free) shared-memory
// accumulators with native shared atomics; the token-MLP weight gradients (contraction over the lanes' hidden
// columns) use a transpose-reduce through shared memory.  One flush of all accumulators per CTA at the end.
#pragma once
#include "mmx_common.cuh"
#include "mmx_mlp.cuh"

namespace mmx {

constexpr int kLPS = 16;   // lanes per sequence
constexpr int kSPW = 2;    // sequences per warp
constexpr int kAccP = 64;  // pitch of the swizzled dV accumulators
constexpr int kRedP = 36;  // row pitch of the per-warp reduction exchange [value][lane]: 4 (mod 32), so the 8 lanes of a
                           // quarter-warp that read 8 different values' rows with 128-bit loads hit 8 different bank groups
                           // (pitch 32 made every such load an 8-way conflict: ncu, 35-46 % of the shared wavefronts)

template <int TC>
struct WLane {
    float a[TC][4], b[TC][4], c[TC][4], e[TC][4];   // register tiles: own 4 hidden columns x T frames
    float rv[2 * TC];                               // row-reduction inputs / totals
    float mu[TC], rs[TC];                           // LayerNorm statistics of the lane's sequence
};

struct MlpWarpSmem {
    int P, PH, PC, TP, KP;
    int ln1_g, ln1_b, ln2_g, ln2_b, cb1, cb2, tw1, tb1, tw2t, tb2, se1, se2, v1, v2;
    int a_v1, a_v2, lock;                     // CTA-shared dV1 / dV2 accumulators (swizzled) + their locks (backward)
    int warp0, wstride;                       // per-warp scratch: base of warp 0, stride between warps
    int tile[3], red, tot, mean1, rstd1, pool1, gate1, z1;   // offsets inside a warp's scratch
    int wv, wtok, wtb2, wse;                  // per-warp PRIVATE gradient accumulators (backward): no atomics needed
    int nse;                                  // floats per SE weight matrix (T * rr)
    int total;
};

constexpr int kTrP = 36;   // row pitch of the token transpose buffers (conflict-free float4 row reads by 8 lanes)

MMX_HD MlpWarpSmem mlp_warp_smem(const MlpDims& d, bool bwd, int nwarp) {
    MlpWarpSmem L;
    const int T = d.T, H = d.H, tok = d.tok, ch = d.ch, rr = imax(d.rr, 1);
    L.P = round_up(imax(H, ch), 4);
    L.PH = pitch_of(H); L.PC = pitch_of(ch);
    L.TP = round_up(T, 4); L.KP = round_up(tok, 4);
    L.nse = T * rr;
    int o = 0;
    auto take = [&](int n) { int r = o; o += round_up(n, 4); return r; };
    L.ln1_g = take(64); L.ln1_b = take(64); L.ln2_g = take(64); L.ln2_b = take(64); L.cb1 = take(64); L.cb2 = take(64);
    L.tw1 = take(tok * L.TP); L.tb1 = take(tok); L.tw2t = take(tok * L.TP); L.tb2 = take(L.TP);
    L.se1 = take(rr * T); L.se2 = take(T * rr);
    L.v1 = take(ch * L.PH); L.v2 = take(H * L.PC);
    if (bwd) { L.a_v1 = take(64 * kAccP); L.a_v2 = take(64 * kAccP); L.lock = take(4); }   // locks: dV1 pass 0/1, dV2 pass 0/1
    else L.a_v1 = L.a_v2 = L.lock = -1;
    L.warp0 = o;
    int w = 0;
    auto wtake = [&](int n) { int r = w; w += round_up(n, 4); return r; };
    const int ntile = bwd ? 3 : 2;
    int tsz = kSPW * T * L.P;
    if (bwd) tsz = imax(tsz, (2 * T + 1) * kTrP);   // tiles 1..2 double as the two token transpose buffers
    for (int i = 0; i < 3; ++i) L.tile[i] = i < ntile ? wtake(tsz) : -1;
    L.red = wtake((bwd ? 2 : 1) * T * kRedP);   // [value][lane]; the backward's transpose buffers (2 x 21 x kTrP) alias tile[1..2]
    L.tot = wtake(kSPW * 2 * T);
    L.mean1 = wtake(kSPW * 16); L.rstd1 = wtake(kSPW * 16); L.pool1 = wtake(kSPW * 16); L.gate1 = wtake(kSPW * 16);
    L.z1 = wtake(kSPW * 16);
    if (bwd) {
        L.wv = wtake(kSPW * 6 * 64);          // [half][ln1g, ln1b, ln2g, ln2b, cb1, cb2][64]
        L.wtok = wtake((2 * T + 1) * tok);    // [dW2[t][.] (T rows), dW1[.][t] (T rows), db1][tok]
        L.wtb2 = wtake(kSPW * 16);
        L.wse = wtake(kSPW * 2 * L.nse);      // [half][dS1, dS2][T*rr]
    } else L.wv = L.wtok = L.wtb2 = L.wse = -1;
    L.wstride = w;
    L.total = o + nwarp * w + 64;       // slack: the outer-product GEMM reads up to 12 floats past a tile row
    return L;
}

// ------------------------------------------------------------------------------------------
// per-warp row reductions across the 16 lanes of each sequence (through shared memory)
// ------------------------------------------------------------------------------------------
template <int NR>
MMX_D void red_write(float* red, int lane, const float* rv) {
    MMX_UNROLL
    for (int r = 0; r < NR; ++r) red[r * kRedP + lane] = rv[r];
}
template <int NR>
MMX_D void red_sum(const float* red, float* tot, int lane) {
    for (int i = lane; i < kSPW * NR; i += 32) {
        const int s = i / NR, r = i - s * NR;
        const float* p = red + r * kRedP + s * kLPS;
        const f4 v0 = ld4(p), v1 = ld4(p + 4), v2 = ld4(p + 8), v3 = ld4(p + 12);
        tot[i] = (((v0.x + v0.y) + (v0.z + v0.w)) + ((v1.x + v1.y) + (v1.z + v1.w))) +
                 (((v2.x + v2.y) + (v2.z + v2.w)) + ((v3.x + v3.y) + (v3.z + v3.w)));
    }
}
template <int NR>
MMX_D void red_read(const float* tot, int s, float* rv) {
    MMX_UNROLL
    for (int r = 0; r < NR; ++r) rv[r] = tot[s * NR + r];
}

// first N floats of a 16-byte aligned shared row (padded to a multiple of 4) into registers, 128 bits at a time
template <int N>
MMX_D void load_row(const float* p, float (&v)[N + 3]) {
    MMX_UNROLL
    for (int i = 0; i < (N + 3) / 4; ++i) { const f4 t = ld4(p + 4 * i); v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w; }
}

// 4 consecutive floats of a global row whose start is only guaranteed 4-byte aligned; n = valid count (0..4)
MMX_D void ldg_row4(const float* p, int n, bool vec, float (&v)[4]) {
    if (vec && n == 4) { const f4 t = ld4(p); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; return; }
    MMX_UNROLL
    for (int j = 0; j < 4; ++j) v[j] = j < n ? p[j] : 0.0f;
}
MMX_D void stg_row4(float* p, int n, bool vec, const float (&v)[4]) {
    if (vec && n == 4) { st4(p, make_f4(v[0], v[1], v[2], v[3])); return; }
    MMX_UNROLL
    for (int j = 0; j < 4; ++j)
        if (j < n) p[j] = v[j];
}

// acc[t][j] += sum_k A[t][k] * W[min(4q+j, N-1)][k]      (NT: W rows are k-contiguous, zero padded to 4)
template <int TC>
MMX_D void warp_gemm_nt(float (&acc)[TC][4], const float* A, int P, const float* W, int ldw, int N, int K, int q) {
    const float* wp[4];
    MMX_UNROLL
    for (int j = 0; j < 4; ++j) wp[j] = W + (size_t)imin(4 * q + j, N - 1) * ldw;
    const int K4 = (K + 3) >> 2;
    MMX_NOUNROLL
    for (int k4 = 0; k4 < K4; ++k4) {
        f4 w[4];
        MMX_UNROLL
        for (int j = 0; j < 4; ++j) w[j] = ld4(wp[j] + 4 * k4);
        MMX_UNROLL
        for (int t = 0; t < TC; ++t) {
            const f4 av = ld4(A + t * P + 4 * k4);
            MMX_UNROLL
            for (int j = 0; j < 4; ++j) {
                acc[t][j] = fmaf(av.x, w[j].x, acc[t][j]); acc[t][j] = fmaf(av.y, w[j].y, acc[t][j]);
                acc[t][j] = fmaf(av.z, w[j].z, acc[t][j]); acc[t][j] = fmaf(av.w, w[j].w, acc[t][j]);
            }
        }
    }
}

// acc[t][j] += sum_{k<K} A[t][k] * W[k][4q+j]            (NN: W is k-major with pitch ldw >= round_up(N,4))
template <int TC>
MMX_D void warp_gemm_nn(float (&acc)[TC][4], const float* A, int P, const float* W, int ldw, int K, int q) {
    const int c0 = 4 * q + 4 <= ldw ? 4 * q : 0;   // lanes past the matrix compute garbage that is never used
    const int K4 = (K + 3) >> 2;
    MMX_NOUNROLL
    for (int k4 = 0; k4 < K4; ++k4) {
        f4 w[4];
        MMX_UNROLL
        for (int i = 0; i < 4; ++i) w[i] = ld4(W + (size_t)imin(4 * k4 + i, K - 1) * ldw + c0);
        MMX_UNROLL
        for (int t = 0; t < TC; ++t) {
            f4 av = ld4(A + t * P + 4 * k4);
            if (4 * k4 + 3 >= K) {   // K tail: the clamped W rows must not contribute
                if (4 * k4 + 1 >= K) av.y = 0.0f;
                if (4 * k4 + 2 >= K) av.z = 0.0f;
                av.w = 0.0f;
            }
            acc[t][0] = fmaf(av.x, w[0].x, acc[t][0]); acc[t][1] = fmaf(av.x, w[0].y, acc[t][1]);
            acc[t][2] = fmaf(av.x, w[0].z, acc[t][2]); acc[t][3] = fmaf(av.x, w[0].w, acc[t][3]);
            acc[t][0] = fmaf(av.y, w[1].x, acc[t][0]); acc[t][1] = fmaf(av.y, w[1].y, acc[t][1]);
            acc[t][2] = fmaf(av.y, w[1].z, acc[t][2]); acc[t][3] = fmaf(av.y, w[1].w, acc[t][3]);
            acc[t][0] = fmaf(av.z, w[2].x, acc[t][0]); acc[t][1] = fmaf(av.z, w[2].y, acc[t][1]);
            acc[t][2] = fmaf(av.z, w[2].z, acc[t][2]); acc[t][3] = fmaf(av.z, w[2].w, acc[t][3]);
            acc[t][0] = fmaf(av.w, w[3].x, acc[t][0]); acc[t][1] = fmaf(av.w, w[3].y, acc[t][1]);
            acc[t][2] = fmaf(av.w, w[3].z, acc[t][2]); acc[t][3] = fmaf(av.w, w[3].w, acc[t][3]);
        }
    }
}

// out[r][c] += sum_{s,t} A[s][t][r] * B[s][t][c]  for r < RA, c < CB, accumulated into a CTA-shared [64][kAccP]
// shared-memory matrix.  Lane (lr, lc) computes rows 8lr..8lr+7 x columns 16lc+8*pass..+7 in registers, then the warp
// takes the matrix lock and adds its tiles with plain 128-bit read-modify-writes.  Quad qd of row r lives at quad
// qd ^ (2*((r>>3)&7)) so the 8 row-groups of a warp spread over the banks.
MMX_D int acc_sw(int r, int c) { return r * kAccP + ((((c >> 2) ^ (((r >> 3) & 7) << 1)) << 2) | (c & 3)); }

template <int TC>
MMX_D void warp_wgrad(float* accm, unsigned int* lock, const float* At, const float* Bt, int P, int RA, int CB, int lane,
                      bool live0, bool live1, int first) {
    const int lr = lane >> 2, lc = lane & 3, r0 = 8 * lr;
    MMX_NOUNROLL
    for (int pp = 0; pp < 2; ++pp) {
        const int pass = pp ^ (first & 1);      // odd warps take the column halves (and their locks) in the other order
        const int c0 = 16 * lc + 8 * pass;
        const bool work = r0 < RA && c0 < CB;
        float acc[8][8];
        MMX_UNROLL
        for (int i = 0; i < 8; ++i)
            MMX_UNROLL
            for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;
        if (work) {
            MMX_NOUNROLL
            for (int s = 0; s < kSPW; ++s) {
                if (!(s == 0 ? live0 : live1)) continue;
                MMX_NOUNROLL
                for (int t = 0; t < TC; ++t) {
                    const float* ar = At + (s * TC + t) * P + r0;
                    const float* br = Bt + (s * TC + t) * P + c0;
                    const f4 a0 = ld4(ar), a1 = ld4(ar + 4), b0 = ld4(br), b1 = ld4(br + 4);
                    const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
                    const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
                    MMX_UNROLL
                    for (int i = 0; i < 8; ++i)
                        MMX_UNROLL
                        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
                }
            }
        }
        warp_lock(lock + pass, lane);      // one lock per (matrix, column half): the two passes touch disjoint columns
        if (work) {
            MMX_UNROLL
            for (int i = 0; i < 8; ++i) {
                if (r0 + i < RA) {      // rows past RA hold garbage (operand columns beyond the tile pitch)
                    float* p0 = accm + acc_sw(r0 + i, c0);
                    float* p1 = accm + acc_sw(r0 + i, c0 + 4);
                    f4 v0 = ld4(p0), v1 = ld4(p1);
                    v0.x += acc[i][0]; v0.y += acc[i][1]; v0.z += acc[i][2]; v0.w += acc[i][3];
                    v1.x += acc[i][4]; v1.y += acc[i][5]; v1.z += acc[i][6]; v1.w += acc[i][7];
                    st4(p0, v0); st4(p1, v1);      // columns past CB accumulate garbage that is never flushed
                }
            }
        }
        warp_unlock(lock + pass, lane);
    }
}

// SE excitation for every frame of one sequence, computed redundantly by each of its lanes:
// z[j] = S1[j,:] . pool ;  gate[t] = sigmoid(S2[t,:] . relu(z))
template <int TC>
MMX_D void se_gates(const float* se1, const float* se2, const float (&pool)[TC], int rr, float (&gate)[TC], float* z /*[rr<=TC]*/) {
    MMX_UNROLL
    for (int t = 0; t < TC; ++t) gate[t] = 0.0f;
    MMX_NOUNROLL
    for (int j = 0; j < rr; ++j) {
        float zz = 0.0f;
        MMX_UNROLL
        for (int t = 0; t < TC; ++t) zz = fmaf(se1[j * TC + t], pool[t], zz);
        z[j] = zz;
        const float rz = fmaxf(zz, 0.0f);
        MMX_UNROLL
        for (int t = 0; t < TC; ++t) gate[t] = fmaf(se2[t * rr + j], rz, gate[t]);
    }
    MMX_UNROLL
    for (int t = 0; t < TC; ++t) gate[t] = sigmoidf_(gate[t]);
}

// SE backward for one sequence (redundant per lane): in dg[t] = sum_h dOut*Y; out ds[t] (gradient of the pooled mean,
// before the 1/H).  When `accumulate` (ONE lane per live sequence) the SE weight gradients are added to that sequence
// slot's private accumulators (plain adds).
template <int TC>
MMX_D void se_backward(const float* se1, const float* se2, const float (&pool)[TC], const float (&gate)[TC], const float* z,
                       int rr, const float (&dg)[TC], float (&ds)[TC], bool accumulate, float* a_se1, float* a_se2) {
    float dq[TC];
    MMX_UNROLL
    for (int t = 0; t < TC; ++t) { dq[t] = dg[t] * gate[t] * (1.0f - gate[t]); ds[t] = 0.0f; }
    MMX_NOUNROLL
    for (int j = 0; j < rr; ++j) {
        float da = 0.0f;
        MMX_UNROLL
        for (int t = 0; t < TC; ++t) da = fmaf(se2[t * rr + j], dq[t], da);
        const float dz = z[j] > 0.0f ? da : 0.0f;
        const float rz = fmaxf(z[j], 0.0f);
        MMX_UNROLL
        for (int t = 0; t < TC; ++t) {
            ds[t] = fmaf(se1[j * TC + t], dz, ds[t]);
            if (accumulate) { a_se2[t * rr + j] += dq[t] * rz; a_se1[j * TC + t] += dz * pool[t]; }
        }
    }
}

MMX_D void mlp_warp_stage(int tid, int nthr, float* sm, const MlpWarpSmem& L, const MlpDims& d, const MlpBlockW& w) {
    const int T = d.T, H = d.H, tok = d.tok, ch = d.ch, rr = d.rr;
    for (int i = tid; i < 64; i += nthr) {
        sm[L.ln1_g + i] = i < H ? w.ln1_g[i] : 0.0f; sm[L.ln1_b + i] = i < H ? w.ln1_b[i] : 0.0f;
        sm[L.ln2_g + i] = i < H ? w.ln2_g[i] : 0.0f; sm[L.ln2_b + i] = i < H ? w.ln2_b[i] : 0.0f;
        sm[L.cb1 + i] = i < ch ? w.cb1[i] : 0.0f; sm[L.cb2 + i] = i < H ? w.cb2[i] : 0.0f;
    }
    for (int i = tid; i < tok * L.TP; i += nthr) {
        const int k = i / L.TP, t = i - k * L.TP;
        sm[L.tw1 + i] = t < T ? w.tw1[k * T + t] : 0.0f;      // W1[k][t]
        sm[L.tw2t + i] = t < T ? w.tw2[t * tok + k] : 0.0f;   // W2[t][k] transposed
    }
    copy_vec(tid, nthr, sm + L.tb1, w.tb1, tok);
    for (int i = tid; i < L.TP; i += nthr) sm[L.tb2 + i] = i < T ? w.tb2[i] : 0.0f;
    if (d.use_se) { copy_vec(tid, nthr, sm + L.se1, w.se1, rr * T); copy_vec(tid, nthr, sm + L.se2, w.se2, T * rr); }
    stage_matrix(tid, nthr, sm + L.v1, w.cw1, ch, H, L.PH);
    stage_matrix(tid, nthr, sm + L.v2, w.cw2, H, ch, L.PC);
}

// token-mixing MLP forward on the lane's 4 columns:  y[t][j] = mask1 * (b2[t] + sum_k W2[t][k] * mask0 * act(b1[k] + W1[k,:] . n[:,j]))
// n: normalised input tile (0 in invalid columns); the result of an invalid column is forced to 0.
template <int ACT, int TC, int TOKC>
MMX_D void token_mlp_fwd(const float* sm, const MlpWarpSmem& L, const float (&n)[TC][4], float (&y)[TC][4], int nvalid,
                         bool drop, const Dropout& dr, int site_base, long long seq, int q, int H4) {
    MMX_UNROLL
    for (int t = 0; t < TC; ++t) {
        const float b2 = sm[L.tb2 + t];
        MMX_UNROLL
        for (int j = 0; j < 4; ++j) y[t][j] = b2;
    }
    float kA[4] = {1.0f, 1.0f, 1.0f, 1.0f}, kB[4] = {1.0f, 1.0f, 1.0f, 1.0f};
    MMX_NOUNROLL
    for (int k = 0; k < TOKC; ++k) {
        float w1[TC + 3], w2[TC + 3];
        load_row<TC>(sm + L.tw1 + k * L.TP, w1); load_row<TC>(sm + L.tw2t + k * L.TP, w2);
        if (drop && !(k & 1)) dropout_rowpair(dr, site_base + 0, (uint64_t)seq * ((TOKC + 1) / 2) + (k >> 1), q, H4, kA, kB);
        float ks[4];
        MMX_UNROLL
        for (int j = 0; j < 4; ++j) ks[j] = (k & 1) ? kB[j] : kA[j];
        const float b1 = sm[L.tb1 + k];
        MMX_UNROLL
        for (int j = 0; j < 4; ++j) {
            float u = b1, u2 = 0.0f;      // two partial sums: shorter dependent FMA chains
            MMX_UNROLL
            for (int t = 0; t + 1 < TC; t += 2) { u = fmaf(w1[t], n[t][j], u); u2 = fmaf(w1[t + 1], n[t + 1][j], u2); }
            if (TC & 1) u = fmaf(w1[TC - 1], n[TC - 1][j], u);
            u += u2;
            const float g = act_fwd<ACT>(u) * ks[j];
            MMX_UNROLL
            for (int t = 0; t < TC; ++t) y[t][j] = fmaf(w2[t], g, y[t][j]);
        }
    }
    float ksA[4] = {1.0f, 1.0f, 1.0f, 1.0f}, ksB[4] = {1.0f, 1.0f, 1.0f, 1.0f};
    MMX_UNROLL
    for (int t = 0; t < TC; ++t) {
        if (drop && !(t & 1)) dropout_rowpair(dr, site_base + 1, (uint64_t)seq * ((TC + 1) / 2) + (t >> 1), q, H4, ksA, ksB);
        const float (&ks)[4] = (t & 1) ? ksB : ksA;
        MMX_UNROLL
        for (int j = 0; j < 4; ++j) y[t][j] = j < nvalid ? y[t][j] * ks[j] : 0.0f;
    }
}

// ------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------
template <int ACT, int TC, int TOKC>
MMX_D void mlp_block_fwd_warp_body(Exec& ex, const MlpBlockFwdArgs& a) {
    const MlpDims& d = a.d;
    float* sm = ex.smem;
    const int nthr = ex.nthr, nwarp = nthr / 32;
    const MlpWarpSmem L = mlp_warp_smem(d, false, nwarp);
    const int H = d.H, ch = d.ch, rr = d.rr, P = L.P;
    const int H4 = (H + 3) >> 2, C4 = (ch + 3) >> 2;
    const float invH = 1.0f / (float)H;
    const bool vecH = (H & 3) == 0;
    const Dropout dr = resolve_dropout(a.dr);
    const bool drop = d.training && dr.thresh != 0u;
    typedef WLane<TC> ST;
    PerThread<ST> regs(ex);

    ex.phase([&](int tid) { mlp_warp_stage(tid, nthr, sm, L, d, a.w); });

    const int groups = (d.B + kSPW - 1) / kSPW;
    ex.warps([&](WarpExec& wx) {
        float* ws = sm + L.warp0 + wx.warp * L.wstride;
        float* red = ws + L.red;
        float* tot = ws + L.tot;
        // every warp of the CTA runs the same number of iterations (a warp without a pair runs a dead one: nothing is stored
        // or accumulated) and the CTA re-aligns once per iteration at wx.align(): the loop body is several times the size of
        // the instruction caches, and warps that walk it together share each fetched line.  The forward time is the same for
        // every choice of re-alignment points (profiles/r1zc_alignment_sweeps.txt); this one sits in front of the X1 phase
        const int per_iter = ex.nblk * nwarp, n_iter = (groups + per_iter - 1) / per_iter;
        for (int it = 0; it < n_iter; ++it) {
            const int grp = it * per_iter + ex.bid * nwarp + wx.warp;
            // lane geometry (recomputed inside each sub-phase from `lane`)
#define MMX_LANE_GEOM                                                                                     \
    ST& st = regs[wx.warp * 32 + lane];                                                                   \
    const int s = lane >> 4, q = lane & 15;                                                               \
    const long long seq_raw = (long long)grp * kSPW + s;                                                  \
    const bool live = seq_raw < d.B;                                                                      \
    const long long seq = live ? seq_raw : d.B - 1;                                                       \
    const int nvh = imax(0, imin(4, H - 4 * q)), nvc = imax(0, imin(4, ch - 4 * q));                      \
    (void)live; (void)nvc; (void)nvh; (void)seq;
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                const float* xg = a.x + (size_t)seq * TC * H + 4 * q;
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    ldg_row4(xg + (size_t)t * H, nvh, vecH, st.a[t]);
                    st.rv[t] = (st.a[t][0] + st.a[t][1]) + (st.a[t][2] + st.a[t][3]);
                }
                red_write<TC>(red, lane, st.rv);
            });
            wx.phase([&](int lane) { red_sum<TC>(red, tot, lane); });
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                red_read<TC>(tot, s, st.rv);
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    st.mu[t] = st.rv[t] * invH;
                    float ss = 0.0f;
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j)
                        if (j < nvh) { const float dv = st.a[t][j] - st.mu[t]; ss = fmaf(dv, dv, ss); }
                    st.rv[t] = ss;
                }
                red_write<TC>(red, lane, st.rv);
            });
            wx.phase([&](int lane) { red_sum<TC>(red, tot, lane); });
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                red_read<TC>(tot, s, st.rv);
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    st.rs[t] = 1.0f / sqrtf(st.rv[t] * invH + 1e-5f);
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j)
                        st.b[t][j] = j < nvh ? (st.a[t][j] - st.mu[t]) * st.rs[t] * sm[L.ln1_g + 4 * q + j] + sm[L.ln1_b + 4 * q + j] : 0.0f;
                }
                token_mlp_fwd<ACT, TC, TOKC>(sm, L, st.b, st.c, nvh, drop, dr, d.site_base, seq, q, H4);
                if (d.use_se) {
                    MMX_UNROLL
                    for (int t = 0; t < TC; ++t) st.rv[t] = (st.c[t][0] + st.c[t][1]) + (st.c[t][2] + st.c[t][3]);
                    red_write<TC>(red, lane, st.rv);
                }
            });
            if (d.use_se) wx.phase([&](int lane) { red_sum<TC>(red, tot, lane); });
            // X1 = X + gate1 * Yt ; LN2 statistics
            wx.align();
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                float gate[TC];
                if (d.use_se) {
                    red_read<TC>(tot, s, st.rv);
                    float pool[TC], z[TC];
                    MMX_UNROLL
                    for (int t = 0; t < TC; ++t) pool[t] = st.rv[t] * invH;
                    se_gates<TC>(sm + L.se1, sm + L.se2, pool, rr, gate, z);
                } else {
                    MMX_UNROLL
                    for (int t = 0; t < TC; ++t) gate[t] = 1.0f;
                }
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j) st.a[t][j] = fmaf(gate[t], st.c[t][j], st.a[t][j]);
                    st.rv[t] = (st.a[t][0] + st.a[t][1]) + (st.a[t][2] + st.a[t][3]);
                }
                red_write<TC>(red, lane, st.rv);
            });
            wx.phase([&](int lane) { red_sum<TC>(red, tot, lane); });
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                red_read<TC>(tot, s, st.rv);
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    st.mu[t] = st.rv[t] * invH;
                    float ss = 0.0f;
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j)
                        if (j < nvh) { const float dv = st.a[t][j] - st.mu[t]; ss = fmaf(dv, dv, ss); }
                    st.rv[t] = ss;
                }
                red_write<TC>(red, lane, st.rv);
            });
            wx.phase([&](int lane) { red_sum<TC>(red, tot, lane); });
            // N2 = LN2(X1) -> tile0
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                red_read<TC>(tot, s, st.rv);
                float* t0 = ws + L.tile[0] + s * TC * P + 4 * q;
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    st.rs[t] = 1.0f / sqrtf(st.rv[t] * invH + 1e-5f);
                    float v[4];
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j)
                        v[j] = j < nvh ? (st.a[t][j] - st.mu[t]) * st.rs[t] * sm[L.ln2_g + 4 * q + j] + sm[L.ln2_b + 4 * q + j] : 0.0f;
                    if (4 * q < P) st4(t0 + t * P, make_f4(v[0], v[1], v[2], v[3]));
                }
            });
            // G2 = drop(act(N2 V1^T + c1)) -> tile1
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                MMX_UNROLL
                for (int t = 0; t < TC; ++t)
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j) st.b[t][j] = 0.0f;
                warp_gemm_nt<TC>(st.b, ws + L.tile[0] + s * TC * P, P, sm + L.v1, L.PH, ch, H, q);
                float* t1 = ws + L.tile[1] + s * TC * P + 4 * q;
                float ksA[4] = {1.0f, 1.0f, 1.0f, 1.0f}, ksB[4] = {1.0f, 1.0f, 1.0f, 1.0f};
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    if (drop && !(t & 1)) dropout_rowpair(dr, d.site_base + 2, (uint64_t)seq * ((TC + 1) / 2) + (t >> 1), q, C4, ksA, ksB);
                    const float (&ks)[4] = (t & 1) ? ksB : ksA;
                    float v[4];
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j) v[j] = j < nvc ? act_fwd<ACT>(st.b[t][j] + sm[L.cb1 + 4 * q + j]) * ks[j] : 0.0f;
                    if (4 * q < P) st4(t1 + t * P, make_f4(v[0], v[1], v[2], v[3]));
                }
            });
            // Y2 = drop(G2 V2^T + c2) ; SE2 squeeze
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                MMX_UNROLL
                for (int t = 0; t < TC; ++t)
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j) st.c[t][j] = 0.0f;
                warp_gemm_nt<TC>(st.c, ws + L.tile[1] + s * TC * P, P, sm + L.v2, L.PC, H, ch, q);
                float ksA[4] = {1.0f, 1.0f, 1.0f, 1.0f}, ksB[4] = {1.0f, 1.0f, 1.0f, 1.0f};
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    if (drop && !(t & 1)) dropout_rowpair(dr, d.site_base + 3, (uint64_t)seq * ((TC + 1) / 2) + (t >> 1), q, H4, ksA, ksB);
                    const float (&ks)[4] = (t & 1) ? ksB : ksA;
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j) st.c[t][j] = j < nvh ? (st.c[t][j] + sm[L.cb2 + 4 * q + j]) * ks[j] : 0.0f;
                    st.rv[t] = (st.c[t][0] + st.c[t][1]) + (st.c[t][2] + st.c[t][3]);
                }
                if (d.use_se) red_write<TC>(red, lane, st.rv);
            });
            if (d.use_se) wx.phase([&](int lane) { red_sum<TC>(red, tot, lane); });
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                float gate[TC];
                if (d.use_se) {
                    red_read<TC>(tot, s, st.rv);
                    float pool[TC], z[TC];
                    MMX_UNROLL
                    for (int t = 0; t < TC; ++t) pool[t] = st.rv[t] * invH;
                    se_gates<TC>(sm + L.se1, sm + L.se2, pool, rr, gate, z);
                } else {
                    MMX_UNROLL
                    for (int t = 0; t < TC; ++t) gate[t] = 1.0f;
                }
                if (live) {
                    float* yg = a.y + (size_t)seq * TC * H + 4 * q;
                    MMX_UNROLL
                    for (int t = 0; t < TC; ++t) {
                        float v[4];
                        MMX_UNROLL
                        for (int j = 0; j < 4; ++j) v[j] = fmaf(gate[t], st.c[t][j], st.a[t][j]);
                        stg_row4(yg + (size_t)t * H, nvh, vecH, v);
                    }
                }
            });
        }
    });
}

// ------------------------------------------------------------------------------------------
// backward (forward recomputed from the block input)
// ------------------------------------------------------------------------------------------
template <int ACT, int TC, int TOKC>
MMX_D void mlp_block_bwd_warp_body(Exec& ex, const MlpBlockBwdArgs& a) {
    const MlpDims& d = a.d;
    float* sm = ex.smem;
    const int nthr = ex.nthr, nwarp = nthr / 32;
    const MlpWarpSmem L = mlp_warp_smem(d, true, nwarp);
    const int H = d.H, ch = d.ch, rr = d.rr, P = L.P;
    const int H4 = (H + 3) >> 2, C4 = (ch + 3) >> 2;
    const float invH = 1.0f / (float)H;
    const bool vecH = (H & 3) == 0;
    const Dropout dr = resolve_dropout(a.dr);
    const bool drop = d.training && dr.thresh != 0u;
    constexpr int NTR = 2 * TC + 1;      // per-k transpose-reduce values: dW2[:,k] (TC), dW1[k,:] (TC), db1[k]
    typedef WLane<TC> ST;
    PerThread<ST> regs(ex);

    ex.phase([&](int tid) {
        mlp_warp_stage(tid, nthr, sm, L, d, a.w);
        for (int i = tid; i < L.total - L.a_v1; i += nthr) sm[L.a_v1 + i] = 0.0f;   // every accumulator (CTA-shared and per-warp), locks
    });

    const int groups = (d.B + kSPW - 1) / kSPW;
    ex.warps([&](WarpExec& wx) {
        float* ws = sm + L.warp0 + wx.warp * L.wstride;
        float* red = ws + L.red;
        float* tot = ws + L.tot;
        float* trb = ws + L.tile[1];     // token phase: 2 transpose buffers [NTR][kTrP] (tiles 1..2 are free by then)
        unsigned int* locks = reinterpret_cast<unsigned int*>(sm + L.lock);
        // every warp of the CTA runs the same number of iterations (a warp without a pair runs a dead one: nothing is stored
        // or accumulated) and the CTA re-aligns once per iteration at wx.align(): the loop body is several times the size of
        // the instruction caches, and warps that walk it together share each fetched line.  Where is a measured choice
        // (profiles/r1zc_alignment_sweeps.txt): after the lock-protected weight-gradient phases is best (backward
        // 316 -> 233 us at B=4096); aligning right in front of those phases makes every warp hit the locks at once and costs
        // more than it saves
        const int per_iter = ex.nblk * nwarp, n_iter = (groups + per_iter - 1) / per_iter;
        for (int it = 0; it < n_iter; ++it) {
            const int grp = it * per_iter + ex.bid * nwarp + wx.warp;
            // ---------------- recompute: LN1, token MLP, SE1, X1, LN2, channel MLP ----------------
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                const float* xg = a.x + (size_t)seq * TC * H + 4 * q;
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    ldg_row4(xg + (size_t)t * H, nvh, vecH, st.a[t]);
                    st.rv[t] = (st.a[t][0] + st.a[t][1]) + (st.a[t][2] + st.a[t][3]);
                }
                red_write<TC>(red, lane, st.rv);
            });
            wx.phase([&](int lane) { red_sum<TC>(red, tot, lane); });
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                red_read<TC>(tot, s, st.rv);
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    st.mu[t] = st.rv[t] * invH;
                    float ss = 0.0f;
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j)
                        if (j < nvh) { const float dv = st.a[t][j] - st.mu[t]; ss = fmaf(dv, dv, ss); }
                    st.rv[t] = ss;
                }
                red_write<TC>(red, lane, st.rv);
            });
            wx.phase([&](int lane) { red_sum<TC>(red, tot, lane); });
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                red_read<TC>(tot, s, st.rv);
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    st.rs[t] = 1.0f / sqrtf(st.rv[t] * invH + 1e-5f);
                    if (q == 0) { ws[L.mean1 + s * 16 + t] = st.mu[t]; ws[L.rstd1 + s * 16 + t] = st.rs[t]; }
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j)
                        st.b[t][j] = j < nvh ? (st.a[t][j] - st.mu[t]) * st.rs[t] * sm[L.ln1_g + 4 * q + j] + sm[L.ln1_b + 4 * q + j] : 0.0f;
                }
                token_mlp_fwd<ACT, TC, TOKC>(sm, L, st.b, st.c, nvh, drop, dr, d.site_base, seq, q, H4);
                if (d.use_se) {
                    MMX_UNROLL
                    for (int t = 0; t < TC; ++t) st.rv[t] = (st.c[t][0] + st.c[t][1]) + (st.c[t][2] + st.c[t][3]);
                    red_write<TC>(red, lane, st.rv);
                }
            });
            if (d.use_se) wx.phase([&](int lane) { red_sum<TC>(red, tot, lane); });
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                float gate[TC];
                if (d.use_se) {
                    red_read<TC>(tot, s, st.rv);
                    float pool[TC], z[TC];
                    MMX_UNROLL
                    for (int t = 0; t < TC; ++t) pool[t] = st.rv[t] * invH;
                    se_gates<TC>(sm + L.se1, sm + L.se2, pool, rr, gate, z);
                    if (q == 0) {
                        MMX_UNROLL
                        for (int t = 0; t < TC; ++t) { ws[L.pool1 + s * 16 + t] = pool[t]; ws[L.gate1 + s * 16 + t] = gate[t]; }
                        for (int j = 0; j < rr; ++j) ws[L.z1 + s * 16 + j] = z[j];
                    }
                } else {
                    MMX_UNROLL
                    for (int t = 0; t < TC; ++t) gate[t] = 1.0f;
                }
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j) st.a[t][j] = fmaf(gate[t], st.c[t][j], st.a[t][j]);   // X1
                    st.rv[t] = (st.a[t][0] + st.a[t][1]) + (st.a[t][2] + st.a[t][3]);
                }
                red_write<TC>(red, lane, st.rv);
            });
            wx.phase([&](int lane) { red_sum<TC>(red, tot, lane); });
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                red_read<TC>(tot, s, st.rv);
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    st.mu[t] = st.rv[t] * invH;
                    float ss = 0.0f;
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j)
                        if (j < nvh) { const float dv = st.a[t][j] - st.mu[t]; ss = fmaf(dv, dv, ss); }
                    st.rv[t] = ss;
                }
                red_write<TC>(red, lane, st.rv);
            });
            wx.phase([&](int lane) { red_sum<TC>(red, tot, lane); });
            wx.phase([&](int lane) {      // N2 -> tile0
                MMX_LANE_GEOM
                red_read<TC>(tot, s, st.rv);
                float* t0 = ws + L.tile[0] + s * TC * P + 4 * q;
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    st.rs[t] = 1.0f / sqrtf(st.rv[t] * invH + 1e-5f);
                    float v[4];
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j)
                        v[j] = j < nvh ? (st.a[t][j] - st.mu[t]) * st.rs[t] * sm[L.ln2_g + 4 * q + j] + sm[L.ln2_b + 4 * q + j] : 0.0f;
                    if (4 * q < P) st4(t0 + t * P, make_f4(v[0], v[1], v[2], v[3]));
                }
            });
            wx.phase([&](int lane) {      // U2 -> e (registers), G2 -> tile1
                MMX_LANE_GEOM
                MMX_UNROLL
                for (int t = 0; t < TC; ++t)
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j) st.b[t][j] = 0.0f;
                warp_gemm_nt<TC>(st.b, ws + L.tile[0] + s * TC * P, P, sm + L.v1, L.PH, ch, H, q);
                float* t1 = ws + L.tile[1] + s * TC * P + 4 * q;
                float ksA[4] = {1.0f, 1.0f, 1.0f, 1.0f}, ksB[4] = {1.0f, 1.0f, 1.0f, 1.0f};
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    if (drop && !(t & 1)) dropout_rowpair(dr, d.site_base + 2, (uint64_t)seq * ((TC + 1) / 2) + (t >> 1), q, C4, ksA, ksB);
                    const float (&ks)[4] = (t & 1) ? ksB : ksA;
                    float u[4], v[4];
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j) {
                        u[j] = j < nvc ? st.b[t][j] + sm[L.cb1 + 4 * q + j] : 0.0f;
                        v[j] = j < nvc ? act_fwd<ACT>(u[j]) * ks[j] : 0.0f;
                    }
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j) st.e[t][j] = u[j];
                    if (4 * q < P) st4(t1 + t * P, make_f4(v[0], v[1], v[2], v[3]));
                }
            });
            // Y2 ; dOut ; SE2 squeeze + dgate2 partials
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                MMX_UNROLL
                for (int t = 0; t < TC; ++t)
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j) st.c[t][j] = 0.0f;
                warp_gemm_nt<TC>(st.c, ws + L.tile[1] + s * TC * P, P, sm + L.v2, L.PC, H, ch, q);
                const float* dg_ = a.dy + (size_t)seq * TC * H + 4 * q;
                float ksA[4] = {1.0f, 1.0f, 1.0f, 1.0f}, ksB[4] = {1.0f, 1.0f, 1.0f, 1.0f};
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    if (drop && !(t & 1)) dropout_rowpair(dr, d.site_base + 3, (uint64_t)seq * ((TC + 1) / 2) + (t >> 1), q, H4, ksA, ksB);
                    const float (&ks)[4] = (t & 1) ? ksB : ksA;
                    ldg_row4(dg_ + (size_t)t * H, nvh, vecH, st.b[t]);
                    float p1 = 0.0f, p2 = 0.0f;
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j) {
                        st.c[t][j] = j < nvh ? (st.c[t][j] + sm[L.cb2 + 4 * q + j]) * ks[j] : 0.0f;
                        p1 += st.c[t][j]; p2 = fmaf(st.b[t][j], st.c[t][j], p2);
                    }
                    st.rv[t] = p1; st.rv[TC + t] = p2;
                }
                if (d.use_se) red_write<2 * TC>(red, lane, st.rv);
            });
            if (d.use_se) wx.phase([&](int lane) { red_sum<2 * TC>(red, tot, lane); });
            // dY2 = (dOut*gate2 + ds2/H) * mask3 -> tile2 ; dc2
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                float gate[TC], ds[TC];
                if (d.use_se) {
                    red_read<2 * TC>(tot, s, st.rv);
                    float pool[TC], z[TC], dg[TC];
                    MMX_UNROLL
                    for (int t = 0; t < TC; ++t) { pool[t] = st.rv[t] * invH; dg[t] = st.rv[TC + t]; }
                    se_gates<TC>(sm + L.se1, sm + L.se2, pool, rr, gate, z);
                    se_backward<TC>(sm + L.se1, sm + L.se2, pool, gate, z, rr, dg, ds, live && q == 0, ws + L.wse + s * 2 * L.nse, ws + L.wse + s * 2 * L.nse + L.nse);
                } else {
                    MMX_UNROLL
                    for (int t = 0; t < TC; ++t) { gate[t] = 1.0f; ds[t] = 0.0f; }
                }
                float* t3 = ws + L.tile[2] + s * TC * P + 4 * q;
                float cs[4] = {0.0f, 0.0f, 0.0f, 0.0f};
                float ksA[4] = {1.0f, 1.0f, 1.0f, 1.0f}, ksB[4] = {1.0f, 1.0f, 1.0f, 1.0f};
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    if (drop && !(t & 1)) dropout_rowpair(dr, d.site_base + 3, (uint64_t)seq * ((TC + 1) / 2) + (t >> 1), q, H4, ksA, ksB);
                    const float (&ks)[4] = (t & 1) ? ksB : ksA;
                    float v[4];
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j) {
                        v[j] = j < nvh ? fmaf(ds[t], invH, st.b[t][j] * gate[t]) * ks[j] : 0.0f;
                        cs[j] += v[j];
                    }
                    if (4 * q < P) st4(t3 + t * P, make_f4(v[0], v[1], v[2], v[3]));
                }
                if (live) {
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j)
                        if (j < nvh) ws[L.wv + (s * 6 + 5) * 64 + 4 * q + j] += cs[j];
                }
            });
            // dV2[h][c] += dY2^T G2 ; dG2 = dY2 V2
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                const bool live0 = (long long)grp * kSPW < d.B, live1 = (long long)grp * kSPW + 1 < d.B;
                warp_wgrad<TC>(sm + L.a_v2, locks + 2, ws + L.tile[2], ws + L.tile[1], P, H, ch, lane, live0, live1, wx.warp);
                MMX_UNROLL
                for (int t = 0; t < TC; ++t)
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j) st.b[t][j] = 0.0f;
                warp_gemm_nn<TC>(st.b, ws + L.tile[2] + s * TC * P, P, sm + L.v2, L.PC, H, q);
            });
            // dU2 = dG2 * mask2 * act'(U2) -> tile1 ; dc1
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                float* t1 = ws + L.tile[1] + s * TC * P + 4 * q;
                float cs[4] = {0.0f, 0.0f, 0.0f, 0.0f};
                float ksA[4] = {1.0f, 1.0f, 1.0f, 1.0f}, ksB[4] = {1.0f, 1.0f, 1.0f, 1.0f};
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    if (drop && !(t & 1)) dropout_rowpair(dr, d.site_base + 2, (uint64_t)seq * ((TC + 1) / 2) + (t >> 1), q, C4, ksA, ksB);
                    const float (&ks)[4] = (t & 1) ? ksB : ksA;
                    float v[4] = {0.0f, 0.0f, 0.0f, 0.0f};
                    if (4 * q < P) {
                        MMX_UNROLL
                        for (int j = 0; j < 4; ++j) {
                            float av;
                            v[j] = j < nvc ? st.b[t][j] * ks[j] * act_fwd_grad<ACT>(st.e[t][j], &av) : 0.0f;
                            cs[j] += v[j];
                        }
                        st4(t1 + t * P, make_f4(v[0], v[1], v[2], v[3]));
                    }
                }
                if (live) {
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j)
                        if (j < nvc) ws[L.wv + (s * 6 + 4) * 64 + 4 * q + j] += cs[j];
                }
            });
            // dV1[c][h] += dU2^T N2 ; dN2 = dU2 V1 ; LN2 backward partials
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                const bool live0 = (long long)grp * kSPW < d.B, live1 = (long long)grp * kSPW + 1 < d.B;
                warp_wgrad<TC>(sm + L.a_v1, locks + 0, ws + L.tile[1], ws + L.tile[0], P, ch, H, lane, live0, live1, wx.warp);
                MMX_UNROLL
                for (int t = 0; t < TC; ++t)
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j) st.c[t][j] = 0.0f;
                warp_gemm_nn<TC>(st.c, ws + L.tile[1] + s * TC * P, P, sm + L.v1, L.PH, ch, q);
                float sg[4] = {0.0f, 0.0f, 0.0f, 0.0f}, sb[4] = {0.0f, 0.0f, 0.0f, 0.0f};
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    float m1 = 0.0f, m2 = 0.0f;
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j) {
                        if (j < nvh) {
                            const float xh = (st.a[t][j] - st.mu[t]) * st.rs[t];
                            const float dn = st.c[t][j];
                            sg[j] = fmaf(dn, xh, sg[j]); sb[j] += dn;
                            const float dxh = dn * sm[L.ln2_g + 4 * q + j];
                            m1 += dxh; m2 = fmaf(dxh, xh, m2);
                        } else st.c[t][j] = 0.0f;
                    }
                    st.rv[t] = m1; st.rv[TC + t] = m2;
                }
                if (live) {
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j)
                        if (j < nvh) { ws[L.wv + (s * 6 + 2) * 64 + 4 * q + j] += sg[j]; ws[L.wv + (s * 6 + 3) * 64 + 4 * q + j] += sb[j]; }
                }
                red_write<2 * TC>(red, lane, st.rv);
            });
            wx.phase([&](int lane) { red_sum<2 * TC>(red, tot, lane); });
            wx.align();
            // dX1 = dOut + LN2'(dN2) -> e ; token half: reload X, LN1, token forward, dgate1 partials
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                red_read<2 * TC>(tot, s, st.rv);
                const float* dg_ = a.dy + (size_t)seq * TC * H + 4 * q;
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    const float m1 = st.rv[t] * invH, m2 = st.rv[TC + t] * invH;
                    ldg_row4(dg_ + (size_t)t * H, nvh, vecH, st.e[t]);      // dOut again (L2 hit)
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j)
                        if (j < nvh) {
                            const float xh = (st.a[t][j] - st.mu[t]) * st.rs[t];
                            st.e[t][j] += st.rs[t] * (st.c[t][j] * sm[L.ln2_g + 4 * q + j] - m1 - xh * m2);
                        }
                }
                const float* xg = a.x + (size_t)seq * TC * H + 4 * q;
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    ldg_row4(xg + (size_t)t * H, nvh, vecH, st.a[t]);
                    st.mu[t] = ws[L.mean1 + s * 16 + t]; st.rs[t] = ws[L.rstd1 + s * 16 + t];
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j)
                        st.b[t][j] = j < nvh ? (st.a[t][j] - st.mu[t]) * st.rs[t] * sm[L.ln1_g + 4 * q + j] + sm[L.ln1_b + 4 * q + j] : 0.0f;
                }
                token_mlp_fwd<ACT, TC, TOKC>(sm, L, st.b, st.c, nvh, drop, dr, d.site_base, seq, q, H4);
                if (d.use_se) {
                    MMX_UNROLL
                    for (int t = 0; t < TC; ++t) {
                        float p2 = 0.0f;
                        MMX_UNROLL
                        for (int j = 0; j < 4; ++j) p2 = fmaf(st.e[t][j], st.c[t][j], p2);
                        st.rv[t] = p2;
                    }
                    red_write<TC>(red, lane, st.rv);
                }
            });
            if (d.use_se) wx.phase([&](int lane) { red_sum<TC>(red, tot, lane); });
            // dYt = (dX1*gate1 + ds1/H) * mask1 -> c ; db2 partials ; dX1 stashed in tile0 ; dN1 accumulator (a) zeroed
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                float gate[TC], ds[TC];
                if (d.use_se) {
                    red_read<TC>(tot, s, st.rv);
                    float pool[TC], z[TC], dg[TC];
                    MMX_UNROLL
                    for (int t = 0; t < TC; ++t) { pool[t] = ws[L.pool1 + s * 16 + t]; gate[t] = ws[L.gate1 + s * 16 + t]; dg[t] = st.rv[t]; }
                    for (int j = 0; j < rr; ++j) z[j] = ws[L.z1 + s * 16 + j];
                    se_backward<TC>(sm + L.se1, sm + L.se2, pool, gate, z, rr, dg, ds, live && q == 0, ws + L.wse + s * 2 * L.nse, ws + L.wse + s * 2 * L.nse + L.nse);
                } else {
                    MMX_UNROLL
                    for (int t = 0; t < TC; ++t) { gate[t] = 1.0f; ds[t] = 0.0f; }
                }
                float* t0 = ws + L.tile[0] + s * TC * P + 4 * q;
                float ksA[4] = {1.0f, 1.0f, 1.0f, 1.0f}, ksB[4] = {1.0f, 1.0f, 1.0f, 1.0f};
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    if (drop && !(t & 1)) dropout_rowpair(dr, d.site_base + 1, (uint64_t)seq * ((TC + 1) / 2) + (t >> 1), q, H4, ksA, ksB);
                    const float (&ks)[4] = (t & 1) ? ksB : ksA;
                    if (4 * q < P) st4(t0 + t * P, make_f4(st.e[t][0], st.e[t][1], st.e[t][2], st.e[t][3]));
                    float p = 0.0f;
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j) {
                        st.c[t][j] = (j < nvh && live) ? fmaf(ds[t], invH, st.e[t][j] * gate[t]) * ks[j] : 0.0f;
                        p += st.c[t][j];
                        st.a[t][j] = 0.0f;
                    }
                    st.rv[t] = p;
                }
                red_write<TC>(red, lane, st.rv);
            });
            wx.phase([&](int lane) {
                red_sum<TC>(red, tot, lane);
            });
            // token-MLP backward, one hidden unit k per sub-phase; weight-gradient partials (contraction over the lanes'
            // hidden columns) are transposed through shared memory: lane v then owns value v of unit k-1
            MMX_NOUNROLL
            for (int k = 0; k <= TOKC; ++k) {
                wx.phase([&](int lane) {
                    MMX_LANE_GEOM
                    if (k == 0 && q == 0 && live) {      // db2[t] (token fc2 bias): totals of the dYt row sums
                        MMX_UNROLL
                        for (int t = 0; t < TC; ++t) ws[L.wtb2 + s * 16 + t] += tot[s * TC + t];
                    }
                    if (k > 0 && lane < NTR) {           // finish unit k-1
                        const float* p = trb + ((k - 1) & 1) * NTR * kTrP + lane * kTrP;
                        float s0 = 0.0f, s1 = 0.0f;
                        MMX_UNROLL
                        for (int i = 0; i < 8; i += 2) {
                            const f4 v = ld4(p + 4 * i), w = ld4(p + 4 * i + 4);
                            s0 += (v.x + v.y) + (v.z + v.w); s1 += (w.x + w.y) + (w.z + w.w);
                        }
                        ws[L.wtok + lane * TOKC + (k - 1)] += s0 + s1;   // row lane: dW2[t][.] | dW1[.][t] | db1, column k-1
                    }
                    if (k < TOKC) {
                        float w1[TC + 3], w2[TC + 3];
                        load_row<TC>(sm + L.tw1 + k * L.TP, w1); load_row<TC>(sm + L.tw2t + k * L.TP, w2);
                        float ks[4] = {1.0f, 1.0f, 1.0f, 1.0f};
                        if (drop) {
                            float kA[4], kB[4];
                            dropout_rowpair(dr, d.site_base + 0, (uint64_t)seq * ((TOKC + 1) / 2) + (k >> 1), q, H4, kA, kB);
                            MMX_UNROLL
                            for (int j = 0; j < 4; ++j) ks[j] = (k & 1) ? kB[j] : kA[j];
                        }
                        const float b1 = sm[L.tb1 + k];
                        float pw2[TC], pw1[TC], pb1 = 0.0f;
                        MMX_UNROLL
                        for (int t = 0; t < TC; ++t) { pw2[t] = 0.0f; pw1[t] = 0.0f; }
                        MMX_UNROLL
                        for (int j = 0; j < 4; ++j) {
                            float u = b1, u2 = 0.0f, dg = 0.0f, dg2 = 0.0f;      // two partial sums each: shorter FMA chains
                            MMX_UNROLL
                            for (int t = 0; t + 1 < TC; t += 2) {
                                u = fmaf(w1[t], st.b[t][j], u); u2 = fmaf(w1[t + 1], st.b[t + 1][j], u2);
                                dg = fmaf(w2[t], st.c[t][j], dg); dg2 = fmaf(w2[t + 1], st.c[t + 1][j], dg2);
                            }
                            if (TC & 1) { u = fmaf(w1[TC - 1], st.b[TC - 1][j], u); dg = fmaf(w2[TC - 1], st.c[TC - 1][j], dg); }
                            u += u2; dg += dg2;
                            float av;
                            const float gp = act_fwd_grad<ACT>(u, &av);
                            const float g = av * ks[j];
                            const float du = dg * ks[j] * gp;
                            pb1 += du;
                            MMX_UNROLL
                            for (int t = 0; t < TC; ++t) {
                                st.a[t][j] = fmaf(w1[t], du, st.a[t][j]);        // dN1
                                pw2[t] = fmaf(st.c[t][j], g, pw2[t]);
                                pw1[t] = fmaf(du, st.b[t][j], pw1[t]);
                            }
                        }
                        float* o = trb + (k & 1) * NTR * kTrP + lane;
                        MMX_UNROLL
                        for (int t = 0; t < TC; ++t) { o[t * kTrP] = pw2[t]; o[(TC + t) * kTrP] = pw1[t]; }
                        o[2 * TC * kTrP] = pb1;
                    }
                });
            }
            // LN1 backward: dX = dX1 + LN1'(dN1)
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                const float* xg = a.x + (size_t)seq * TC * H + 4 * q;
                float sg[4] = {0.0f, 0.0f, 0.0f, 0.0f}, sb[4] = {0.0f, 0.0f, 0.0f, 0.0f};
                MMX_UNROLL
                for (int t = 0; t < TC; ++t) {
                    ldg_row4(xg + (size_t)t * H, nvh, vecH, st.c[t]);
                    float m1 = 0.0f, m2 = 0.0f;
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j) {
                        if (j < nvh) {
                            const float xh = (st.c[t][j] - st.mu[t]) * st.rs[t];
                            st.c[t][j] = xh;
                            const float dn = st.a[t][j];
                            sg[j] = fmaf(dn, xh, sg[j]); sb[j] += dn;
                            const float dxh = dn * sm[L.ln1_g + 4 * q + j];
                            m1 += dxh; m2 = fmaf(dxh, xh, m2);
                        }
                    }
                    st.rv[t] = m1; st.rv[TC + t] = m2;
                }
                if (live) {
                    MMX_UNROLL
                    for (int j = 0; j < 4; ++j)
                        if (j < nvh) { ws[L.wv + (s * 6 + 0) * 64 + 4 * q + j] += sg[j]; ws[L.wv + (s * 6 + 1) * 64 + 4 * q + j] += sb[j]; }
                }
                red_write<2 * TC>(red, lane, st.rv);
            });
            wx.phase([&](int lane) { red_sum<2 * TC>(red, tot, lane); });
            wx.phase([&](int lane) {
                MMX_LANE_GEOM
                red_read<2 * TC>(tot, s, st.rv);
                if (live && 4 * q < P) {
                    const float* t0 = ws + L.tile[0] + s * TC * P + 4 * q;
                    float* dxg = a.dx + (size_t)seq * TC * H + 4 * q;
                    MMX_UNROLL
                    for (int t = 0; t < TC; ++t) {
                        const float m1 = st.rv[t] * invH, m2 = st.rv[TC + t] * invH;
                        const f4 dd = ld4(t0 + t * P);
                        const float dv[4] = {dd.x, dd.y, dd.z, dd.w};
                        float v[4];
                        MMX_UNROLL
                        for (int j = 0; j < 4; ++j)
                            v[j] = dv[j] + st.rs[t] * (st.a[t][j] * sm[L.ln1_g + 4 * q + j] - m1 - st.c[t][j] * m2);
                        stg_row4(dxg + (size_t)t * H, nvh, vecH, v);
                    }
                }
            });
        }
    });

    // ---------------- flush the CTA's gradient accumulators ----------------
    ex.phase([&](int) {});
    ex.phase([&](int tid) {
        const int T = d.T, tok = d.tok;
        for (int i = tid; i < ch * H; i += nthr) { const int r = i / H, c = i - r * H; red_add(a.g.cw1 + i, sm[L.a_v1 + acc_sw(r, c)]); }   // dV1 [ch][H]
        for (int i = tid; i < H * ch; i += nthr) { const int r = i / ch, c = i - r * ch; red_add(a.g.cw2 + i, sm[L.a_v2 + acc_sw(r, c)]); } // dV2 [H][ch]
        // per-warp private accumulators: summed over the CTA's warps (and sequence slots) by the owning thread, then one RED
        for (int i = tid; i < 6 * 64; i += nthr) {
            const int kind = i >> 6, col = i & 63;
            const int n = kind == 4 ? ch : H;
            if (col >= n) continue;
            float v = 0.0f;
            for (int w = 0; w < nwarp; ++w)
                for (int s = 0; s < kSPW; ++s) v += sm[L.warp0 + w * L.wstride + L.wv + (s * 6 + kind) * 64 + col];
            float* dst = kind == 0 ? a.g.ln1_g : kind == 1 ? a.g.ln1_b : kind == 2 ? a.g.ln2_g : kind == 3 ? a.g.ln2_b : kind == 4 ? a.g.cb1 : a.g.cb2;
            red_add(dst + col, v);
        }
        for (int i = tid; i < (2 * T + 1) * tok; i += nthr) {
            const int row = i / tok, k = i - row * tok;
            float v = 0.0f;
            for (int w = 0; w < nwarp; ++w) v += sm[L.warp0 + w * L.wstride + L.wtok + i];
            if (row < T) red_add(a.g.tw2 + row * tok + k, v);                  // dW2[t][k]
            else if (row < 2 * T) red_add(a.g.tw1 + k * T + (row - T), v);     // dW1[k][t]
            else red_add(a.g.tb1 + k, v);
        }
        for (int t = tid; t < T; t += nthr) {
            float v = 0.0f;
            for (int w = 0; w < nwarp; ++w)
                for (int s = 0; s < kSPW; ++s) v += sm[L.warp0 + w * L.wstride + L.wtb2 + s * 16 + t];
            red_add(a.g.tb2 + t, v);
        }
        if (d.use_se)
            for (int i = tid; i < 2 * L.nse; i += nthr) {
                float v = 0.0f;
                for (int w = 0; w < nwarp; ++w)
                    for (int s = 0; s < kSPW; ++s) v += sm[L.warp0 + w * L.wstride + L.wse + s * 2 * L.nse + i];
                red_add(i < L.nse ? a.g.se1 + i : a.g.se2 + (i - L.nse), v);
            }
    });
}

#undef MMX_LANE_GEOM

}  // namespace mmx
