// MixerBlock on the Blackwell tensor cores: launch layer of the tcgen05 kernel family (mmx_tok.cuh + mmx_chan_tc5.cuh).
// Reached from mmx_mlp_block_fwd / mmx_mlp_block_bwd when MmxMlpBlockDesc.precision == MMX_PREC_TF32 (the reduced-precision,
// 2e-3 mode) and the shape is one this family serves.  A block runs as
//     forward :  token half (x -> x1, written into y)            ->  channel half (y -> y, in place, tile-local)
//     backward:  token half forward (x -> x1, written into dx)   ->  channel half backward (dx = x1, dy -> dx = dx1, in place)
//                                                                ->  token half backward (x, dx = dx1 -> dx, in place)
// so no workspace is needed beyond the caller's output buffer.
#include "mmx_launch.cuh"

#if defined(MMX_HOST_EMU)
bool mmx_mlp_tc5_ok(const MmxMlpBlockDesc*) { return false; }
int mmx_mlp_tc5_fwd(const MmxMlpBlockDesc*, const MmxMlpBlockParams*, const float*, float*, void*) { return fail(MMX_E_UNSUPPORTED, "no tensor cores in the emulator"); }
int mmx_mlp_tc5_bwd(const MmxMlpBlockDesc*, const MmxMlpBlockParams*, const MmxMlpBlockParams*, const float*, const float*, float*, void*) {
    return fail(MMX_E_UNSUPPORTED, "no tensor cores in the emulator");
}
extern "C" int mmx_tc5_abort_count(void) { return 0; }
extern "C" int mmx_tc5_dropout_mask(const MmxDropout*, unsigned int, long long, int, float*, void*) { return fail(MMX_E_UNSUPPORTED, "no tensor cores in the emulator"); }
int mmx_mlp_tc5_fwd_save(const MmxMlpBlockDesc*, const MmxMlpBlockParams*, const float*, float*, float*, float*, void*) { return fail(MMX_E_UNSUPPORTED, "no tensor cores in the emulator"); }
int mmx_mlp_tc5_bwd_saved(const MmxMlpBlockDesc*, const MmxMlpBlockParams*, const MmxMlpBlockParams*, const float*, const float*, const float*, const float*, float*, void*) {
    return fail(MMX_E_UNSUPPORTED, "no tensor cores in the emulator");
}
#else
#include "mmx_chan_tc5.cuh"
#include "mmx_tc5_launch.cuh"
#include "mmx_tok.cuh"

using namespace mmx;

__device__ int g_mmx_tc5_abort = 0;

int* mmx_tc5_abort_ptr() {
    static int* p[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) dev = 0;
    if (!p[dev]) {
        void* q = nullptr;
        cudaGetSymbolAddress(&q, g_mmx_tc5_abort);
        p[dev] = (int*)q;
    }
    return p[dev];
}

// number of kernels of this family whose pipeline waits timed out since the process started (0 in a healthy run); synchronises
extern "C" int mmx_tc5_abort_count(void) {
    int v = 0;
    cudaMemcpy(&v, mmx_tc5_abort_ptr(), sizeof(int), cudaMemcpyDeviceToHost);
    return v;
}

// keep-scales of one dropout site of this kernel family, as the kernels draw them (debug / test entry point)
static __global__ void tc5_mask_kernel(Dropout dr, uint32_t site, long long rows, int W, float* out) {
    const uint32_t key = tc5::drop_key(dr.seed_lo, dr.seed_hi, site, dr.step), W8 = (uint32_t)(W + 7) >> 3;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < rows * W; i += (long long)gridDim.x * blockDim.x) {
        const uint32_t row = (uint32_t)(i / W), w = (uint32_t)(i - (long long)row * W);
        const uint32_t kb = dr.thresh >> 16 ? tc5::keep8(key, dr.thresh >> 16, row, W8, w >> 3) : 0xffu;
        out[i] = (kb >> (w & 7)) & 1u ? dr.scale : 0.0f;
    }
}
extern "C" int mmx_tc5_dropout_mask(const MmxDropout* d, unsigned int site, long long rows, int W, float* out, void* stream) {
    if (!d || !out || rows <= 0 || W <= 0) return fail(MMX_E_INVALID, "mmx_tc5_dropout_mask: bad argument");
    const Dropout dr = make_dropout(*d, 1);
    tc5_mask_kernel<<<256, 256, 0, (cudaStream_t)stream>>>(dr, site, rows, W, out);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(MMX_E_CUDA, "kernel launch: %s", cudaGetErrorString(e));
    return MMX_OK;
}

// defined in mmx_api_mlp_wide.cu: the wide variant of the channel half (80 <= max(H, ch) <= 128, weights streamed from a workspace)
int mmx_chan_wide_run(bool bwd, int act, const void* chan_args, void* stream);

// padded operand width: 64 / 80 (resident weights, bias gradients in a ones column) or 128 (the wide variant); 0: not served
static int kp_of(const MmxMlpBlockDesc* d) {
    const int need = (d->H > d->ch ? d->H : d->ch) + 1;      // + the ones column that carries the bias gradients
    if (need <= 64) return 64;
    if (need <= 80) return 80;
    if (need - 1 <= 128 && !(d->ch & 1)) return 128;
    return 0;
}

bool mmx_mlp_tc5_ok(const MmxMlpBlockDesc* d) {
    if (d->precision != MMX_PREC_TF32) return false;
    if (d->T < 2 || d->T > tok::kMaxT || d->tok < 1 || d->tok > tok::kMaxTok) return false;
    if (d->H < 8 || d->ch < 8 || (d->H & 1) || kp_of(d) == 0) return false;
    if ((d->T * d->H) & 3) return false;                      // bulk copies: every tile is a multiple of 16 bytes
    if (d->use_max_pooling) return false;
    if (d->use_se && (d->se_hidden < 1 || d->se_hidden > chan::kMaxRR)) return false;
    if (d->H > tok::kTokThreads) return false;
    return true;
}

// ------------------------------------------------------------------------------------------ token half
static int tok_S(const MmxMlpBlockDesc* d) {
    int S = imin(tok::kTokThreads / d->H, tok::kTokThreads / d->T);
    if (S < 1) S = 1;
    return S;
}

static void fill_tok(tok::TokArgs& t, const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const MmxMlpBlockParams* g, int S) {
    t.ln_g = w->ln1_w; t.ln_b = w->ln1_b; t.w1 = w->tok_w1; t.b1 = w->tok_b1; t.w2 = w->tok_w2; t.b2 = w->tok_b2;
    t.se1 = w->se_w1; t.se2 = w->se_w2;
    if (g) {
        t.g_ln_g = g->ln1_w; t.g_ln_b = g->ln1_b; t.g_w1 = g->tok_w1; t.g_b1 = g->tok_b1; t.g_w2 = g->tok_w2; t.g_b2 = g->tok_b2;
        t.g_se1 = g->se_w1; t.g_se2 = g->se_w2;
    } else {
        t.g_ln_g = t.g_ln_b = t.g_w1 = t.g_b1 = t.g_w2 = t.g_b2 = t.g_se1 = t.g_se2 = nullptr;
    }
    t.B = d->B; t.T = d->T; t.H = d->H; t.tok = d->tok; t.rr = d->use_se ? d->se_hidden : 0;
    t.gate_out = nullptr; t.x1s = nullptr; t.gates = nullptr;
    t.S = S; t.site_base = d->block_index * 4;
    t.dr = make_dropout(d->dropout, d->training);
    t.abort_count = mmx_tc5_abort_ptr();
}

template <int ACT, int TT>
static int run_tok(bool bwd, const tok::TokArgs& t, void* stream) {
    const DevInfo di = dev_info();
    const tok::TokSmem m = tok::tok_smem(t.T, t.H, t.tok, t.S, TT, bwd);
    const size_t smem = (size_t)m.total * 4;
    if (smem > (size_t)di.max_smem) return fail(MMX_E_UNSUPPORTED, "token half: tile does not fit shared memory (H=%d)", t.H);
    const int threads = tok::kTokThreads;
    int per_sm = (int)((di.max_smem + 1024) / (smem + 1024));
    per_sm = imax(1, imin(per_sm, bwd ? 2 : 4));
    const int ntiles = (t.B + t.S - 1) / t.S;
    const int grid = balanced_grid(ntiles, di.sms * per_sm);
    return bwd ? launch_tc5(tok::tok_bwd_kernel<ACT, TT>, t, grid, threads, smem, stream)
               : launch_tc5(tok::tok_fwd_kernel<ACT, TT>, t, grid, threads, smem, stream);
}

static int tok_dispatch(bool bwd, const MmxMlpBlockDesc* d, const tok::TokArgs& t, void* stream) {
    const bool gelu = d->act == MMX_ACT_GELU;
    if (d->T == 10) return gelu ? run_tok<ACT_GELU, 10>(bwd, t, stream) : run_tok<ACT_MISH, 10>(bwd, t, stream);
    return gelu ? run_tok<ACT_GELU, 16>(bwd, t, stream) : run_tok<ACT_MISH, 16>(bwd, t, stream);
}

// ------------------------------------------------------------------------------------------ channel half
static void fill_chan(chan::ChanArgs& c, const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const MmxMlpBlockParams* g) {
    c.ln_g = w->ln2_w; c.ln_b = w->ln2_b; c.w1 = w->ch_w1; c.b1 = w->ch_b1; c.w2 = w->ch_w2; c.b2 = w->ch_b2;
    c.se1 = w->se_w1; c.se2 = w->se_w2;
    if (g) {
        c.g_ln_g = g->ln2_w; c.g_ln_b = g->ln2_b; c.g_w1 = g->ch_w1; c.g_b1 = g->ch_b1; c.g_w2 = g->ch_w2; c.g_b2 = g->ch_b2;
        c.g_se1 = g->se_w1; c.g_se2 = g->se_w2;
    } else {
        c.g_ln_g = c.g_ln_b = c.g_w1 = c.g_b1 = c.g_w2 = c.g_b2 = c.g_se1 = c.g_se2 = nullptr;
    }
    c.B = d->B; c.T = d->T; c.H = d->H; c.ch = d->ch; c.rr = d->use_se ? d->se_hidden : 0;
    c.site_base = d->block_index * 4;
    c.dr = make_dropout(d->dropout, d->training);
    c.abort_count = mmx_tc5_abort_ptr();
}

template <int ACT, int KP, int VEC>
static int run_chan(bool bwd, const chan::ChanArgs& c, void* stream) {
    const DevInfo di = dev_info();
    const chan::Geo g = chan::make_geo(c.T, c.H, VEC);
    const size_t smem = chan::chan_smem<KP>(g, bwd).total;
    if (smem > (size_t)di.max_smem) return fail(MMX_E_UNSUPPORTED, "channel half: tile does not fit shared memory (H=%d ch=%d)", c.H, c.ch);
    const int ntiles = (c.B + g.seq_per_tile - 1) / g.seq_per_tile;
    // TMEM: forward 2*KP columns (<= 2 CTAs / SM at KP = 64), backward 4*KP columns
    int per_sm = (int)((di.max_smem + 1024) / (smem + 1024));
    const int tm_cols = bwd ? 512 : (3 * KP <= 256 ? 256 : 512);
    per_sm = imax(1, imin(per_sm, 512 / tm_cols));
    const int grid = imin(ntiles, di.sms * per_sm);
    return bwd ? launch_tc5(chan::chan_bwd_kernel<ACT, KP, VEC>, c, grid, tc5::kCtaThreads, smem, stream)
               : launch_tc5(chan::chan_fwd_kernel<ACT, KP, VEC>, c, grid, tc5::kCtaThreads, smem, stream);
}

template <int ACT>
static int chan_dispatch_act(bool bwd, const MmxMlpBlockDesc* d, const chan::ChanArgs& c, void* stream) {
    const int kp = kp_of(d);
    const bool vec4 = (d->H & 3) == 0;
    if (kp == 64) return vec4 ? run_chan<ACT, 64, 4>(bwd, c, stream) : run_chan<ACT, 64, 2>(bwd, c, stream);
    return vec4 ? run_chan<ACT, 80, 4>(bwd, c, stream) : run_chan<ACT, 80, 2>(bwd, c, stream);
}
static int chan_dispatch(bool bwd, const MmxMlpBlockDesc* d, const chan::ChanArgs& c, void* stream) {
    if (kp_of(d) == 128) return mmx_chan_wide_run(bwd, d->act, &c, stream);
    // H, ch <= 64: the streamed-weight design at operand width 64 leaves room for TWO CTAs per SM (256 TMEM columns, < 100 KB
    // shared each, 64 registers).  Measured on B200 (block fwd / bwd, us): B = 4096, H = 50: 46 / 142 resident vs 47 / 154
    // streamed (1.2 tiles per CTA: the second CTA only doubles the per-CTA flush); B = 16384: 138 / 485 vs 138 / 463;
    // H = ch = 64 (operand width 80 in the resident plan): 83 / 215 vs 78 / 205.  So: streamed when the resident plan would
    // need the 80-column operands, or when every CTA slot gets >= 4 tiles.  MMX_CHAN_STREAMED: bit 0 forward, bit 1 backward
    // (default -1 = this policy).
    if (d->H <= 64 && d->ch <= 64 && !(d->ch & 1)) {
        const int forced = env_int("MMX_CHAN_STREAMED", -1);
        const chan::Geo g = chan::make_geo(d->T, d->H, (d->H & 3) ? 2 : 4);
        const int ntiles = (d->B + g.seq_per_tile - 1) / g.seq_per_tile;
        const bool policy = kp_of(d) == 80 || (bwd && ntiles >= 8 * dev_info().sms);
        if (forced >= 0 ? (forced & (bwd ? 2 : 1)) != 0 : policy) return mmx_chan_wide_run(bwd, d->act, &c, stream);
    }
    return d->act == MMX_ACT_GELU ? chan_dispatch_act<ACT_GELU>(bwd, d, c, stream) : chan_dispatch_act<ACT_MISH>(bwd, d, c, stream);
}

static int check_common(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const char* what) {
    if (d->B <= 0) return fail(MMX_E_INVALID, "non-positive dimension");
    if (d->act != MMX_ACT_GELU && d->act != MMX_ACT_MISH) return fail(MMX_E_INVALID, "Unknown activation function type: %d", d->act);
    if (!w) return fail(MMX_E_INVALID, "%s: null parameter table", what);
    const float* v[] = {w->ln1_w, w->ln1_b, w->tok_w1, w->tok_b1, w->tok_w2, w->tok_b2, w->ln2_w, w->ln2_b, w->ch_w1, w->ch_b1, w->ch_w2, w->ch_b2};
    for (const float* q : v)
        if (!q) return fail(MMX_E_INVALID, "%s: null parameter pointer", what);
    if (d->use_se && (!w->se_w1 || !w->se_w2)) return fail(MMX_E_INVALID, "%s: use_se set but SE weights are null", what);
    return MMX_OK;
}

int mmx_mlp_tc5_fwd(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const float* x, float* y, void* stream) {
    int rc = check_common(d, w, "mmx_mlp_block_fwd");
    if (rc) return rc;
    if ((((uintptr_t)x) | ((uintptr_t)y)) & 15) return fail(MMX_E_INVALID, "mmx_mlp_block_fwd: tensors must be 16-byte aligned");
    const int S = tok_S(d);
    tok::TokArgs t;
    fill_tok(t, d, w, nullptr, S);
    t.x = x; t.dx1 = nullptr; t.out = y;
    if ((rc = tok_dispatch(false, d, t, stream))) return rc;
    chan::ChanArgs c;
    fill_chan(c, d, w, nullptr);
    c.x1 = y; c.dy = nullptr; c.out = y;
    return chan_dispatch(false, d, c, stream);
}

// forward that also saves the token-half output x1 [B,T,H] and its SE gates [B,T] (gate may be null without SE) for
// mmx_mlp_tc5_bwd_saved, which then neither re-runs the token half forward nor recomputes the token MLP output
int mmx_mlp_tc5_fwd_save(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const float* x, float* y, float* x1, float* gate, void* stream) {
    int rc = check_common(d, w, "mmx_mlp_block_fwd_save");
    if (rc) return rc;
    if (!x1 || (d->use_se && !gate)) return fail(MMX_E_INVALID, "mmx_mlp_block_fwd_save: null save buffer");
    if ((((uintptr_t)x) | ((uintptr_t)y) | ((uintptr_t)x1)) & 15) return fail(MMX_E_INVALID, "mmx_mlp_block_fwd_save: tensors must be 16-byte aligned");
    const int S = tok_S(d);
    tok::TokArgs t;
    fill_tok(t, d, w, nullptr, S);
    t.x = x; t.dx1 = nullptr; t.out = x1; t.gate_out = d->use_se ? gate : nullptr;
    if ((rc = tok_dispatch(false, d, t, stream))) return rc;
    chan::ChanArgs c;
    fill_chan(c, d, w, nullptr);
    c.x1 = x1; c.dy = nullptr; c.out = y;
    return chan_dispatch(false, d, c, stream);
}

int mmx_mlp_tc5_bwd_saved(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const MmxMlpBlockParams* grads, const float* x,
                          const float* x1, const float* gate, const float* dy, float* dx, void* stream) {
    int rc = check_common(d, w, "mmx_mlp_block_bwd_saved");
    if (rc) return rc;
    if ((rc = check_common(d, grads, "mmx_mlp_block_bwd_saved(grads)"))) return rc;
    if (!x1 || (d->use_se && !gate)) return fail(MMX_E_INVALID, "mmx_mlp_block_bwd_saved: null saved tensor");
    if ((((uintptr_t)x) | ((uintptr_t)dy) | ((uintptr_t)dx) | ((uintptr_t)x1)) & 15) return fail(MMX_E_INVALID, "mmx_mlp_block_bwd_saved: tensors must be 16-byte aligned");
    if (dx == dy || dx == x || dx == x1) return fail(MMX_E_INVALID, "mmx_mlp_block_bwd_saved: dx must not alias an input");
    chan::ChanArgs c;
    fill_chan(c, d, w, grads);
    c.x1 = x1; c.dy = dy; c.out = dx;
    if ((rc = chan_dispatch(true, d, c, stream))) return rc;
    const int S = tok_S(d);
    tok::TokArgs t;
    fill_tok(t, d, w, grads, S);
    t.x = x; t.dx1 = dx; t.out = dx; t.x1s = x1; t.gates = d->use_se ? gate : nullptr;
    return tok_dispatch(true, d, t, stream);
}

int mmx_mlp_tc5_bwd(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const MmxMlpBlockParams* grads, const float* x,
                    const float* dy, float* dx, void* stream) {
    int rc = check_common(d, w, "mmx_mlp_block_bwd");
    if (rc) return rc;
    if ((rc = check_common(d, grads, "mmx_mlp_block_bwd(grads)"))) return rc;
    if ((((uintptr_t)x) | ((uintptr_t)dy) | ((uintptr_t)dx)) & 15) return fail(MMX_E_INVALID, "mmx_mlp_block_bwd: tensors must be 16-byte aligned");
    if (dx == dy || dx == x) return fail(MMX_E_INVALID, "mmx_mlp_block_bwd: dx must not alias x or dy");
    const int S = tok_S(d);
    tok::TokArgs t;
    fill_tok(t, d, w, grads, S);
    t.x = x; t.dx1 = nullptr; t.out = dx;                         // x1 -> dx
    if ((rc = tok_dispatch(false, d, t, stream))) return rc;
    chan::ChanArgs c;
    fill_chan(c, d, w, grads);
    c.x1 = dx; c.dy = dy; c.out = dx;                             // dx1 -> dx (in place)
    if ((rc = chan_dispatch(true, d, c, stream))) return rc;
    t.dx1 = dx; t.out = dx;
    return tok_dispatch(true, d, t, stream);
}
#endif

// ------------------------------------------------------------------------------------------ the two halves as entry points
// (what mmx_mlp_block_{fwd,bwd}[_save[d]] are made of; used by the benchmark to time the dominant kernel on its own)
#if !defined(MMX_HOST_EMU)
extern "C" int mmx_mlp_token_half_fwd(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const float* x, float* x1, float* gate, void* stream) {
    if (!d || !mmx_mlp_tc5_ok(d)) return fail(MMX_E_UNSUPPORTED, "mmx_mlp_token_half_fwd: shape / precision not served by the tcgen05 family");
    int rc = check_common(d, w, "mmx_mlp_token_half_fwd");
    if (rc) return rc;
    if (!x || !x1) return fail(MMX_E_INVALID, "mmx_mlp_token_half_fwd: null tensor");
    tok::TokArgs t;
    fill_tok(t, d, w, nullptr, tok_S(d));
    t.x = x; t.out = x1; t.gate_out = d->use_se ? gate : nullptr;
    return tok_dispatch(false, d, t, stream);
}
extern "C" int mmx_mlp_token_half_bwd(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const MmxMlpBlockParams* grads, const float* x,
                                      const float* x1, const float* gate, const float* dx1, float* dx, void* stream) {
    if (!d || !mmx_mlp_tc5_ok(d)) return fail(MMX_E_UNSUPPORTED, "mmx_mlp_token_half_bwd: shape / precision not served by the tcgen05 family");
    int rc = check_common(d, w, "mmx_mlp_token_half_bwd");
    if (rc) return rc;
    if ((rc = check_common(d, grads, "mmx_mlp_token_half_bwd(grads)"))) return rc;
    if (!x || !dx1 || !dx) return fail(MMX_E_INVALID, "mmx_mlp_token_half_bwd: null tensor");
    tok::TokArgs t;
    fill_tok(t, d, w, grads, tok_S(d));
    t.x = x; t.dx1 = dx1; t.out = dx; t.x1s = x1; t.gates = (x1 && d->use_se) ? gate : nullptr;
    if (t.x1s && d->use_se && !t.gates) return fail(MMX_E_INVALID, "mmx_mlp_token_half_bwd: saved x1 without its gates");
    return tok_dispatch(true, d, t, stream);
}
extern "C" int mmx_mlp_channel_half_fwd(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const float* x1, float* y, void* stream) {
    if (!d || !mmx_mlp_tc5_ok(d)) return fail(MMX_E_UNSUPPORTED, "mmx_mlp_channel_half_fwd: shape / precision not served by the tcgen05 family");
    int rc = check_common(d, w, "mmx_mlp_channel_half_fwd");
    if (rc) return rc;
    if (!x1 || !y) return fail(MMX_E_INVALID, "mmx_mlp_channel_half_fwd: null tensor");
    chan::ChanArgs c;
    fill_chan(c, d, w, nullptr);
    c.x1 = x1; c.dy = nullptr; c.out = y;
    return chan_dispatch(false, d, c, stream);
}
extern "C" int mmx_mlp_channel_half_bwd(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const MmxMlpBlockParams* grads, const float* x1,
                                        const float* dy, float* dx1, void* stream) {
    if (!d || !mmx_mlp_tc5_ok(d)) return fail(MMX_E_UNSUPPORTED, "mmx_mlp_channel_half_bwd: shape / precision not served by the tcgen05 family");
    int rc = check_common(d, w, "mmx_mlp_channel_half_bwd");
    if (rc) return rc;
    if ((rc = check_common(d, grads, "mmx_mlp_channel_half_bwd(grads)"))) return rc;
    if (!x1 || !dy || !dx1) return fail(MMX_E_INVALID, "mmx_mlp_channel_half_bwd: null tensor");
    chan::ChanArgs c;
    fill_chan(c, d, w, grads);
    c.x1 = x1; c.dy = dy; c.out = dx1;
    return chan_dispatch(true, d, c, stream);
}
#else
extern "C" int mmx_mlp_token_half_fwd(const MmxMlpBlockDesc*, const MmxMlpBlockParams*, const float*, float*, float*, void*) { return fail(MMX_E_UNSUPPORTED, "no tensor cores in the emulator"); }
extern "C" int mmx_mlp_token_half_bwd(const MmxMlpBlockDesc*, const MmxMlpBlockParams*, const MmxMlpBlockParams*, const float*, const float*, const float*, const float*, float*, void*) { return fail(MMX_E_UNSUPPORTED, "no tensor cores in the emulator"); }
extern "C" int mmx_mlp_channel_half_fwd(const MmxMlpBlockDesc*, const MmxMlpBlockParams*, const float*, float*, void*) { return fail(MMX_E_UNSUPPORTED, "no tensor cores in the emulator"); }
extern "C" int mmx_mlp_channel_half_bwd(const MmxMlpBlockDesc*, const MmxMlpBlockParams*, const MmxMlpBlockParams*, const float*, const float*, float*, void*) { return fail(MMX_E_UNSUPPORTED, "no tensor cores in the emulator"); }
#endif
