// mmx_pose_encoder_{fwd,bwd}, mmx_conv_head_{fwd,bwd} (include/mmx.h).
#include "mmx_launch.cuh"
#include "mmx_conv_io.cuh"

using namespace mmx;

namespace mmx_tu_conv_io {
struct EncFwdBody { static MMX_D void run(Exec& ex, const EncFwdArgs& a) { enc_fwd_body(ex, a); } };
struct EncBwd1Body { static MMX_D void run(Exec& ex, const EncBwd1Args& a) { enc_bwd1_body(ex, a); } };
struct EncBwd2Body { static MMX_D void run(Exec& ex, const EncBwd2Args& a) { enc_bwd2_body(ex, a); } };
struct HeadFwdBody { static MMX_D void run(Exec& ex, const ConvHeadFwdArgs& a) { conv_head_fwd_body(ex, a); } };
struct HeadFwdChunkBody { static MMX_D void run(Exec& ex, const ConvHeadFwdArgs& a) { conv_head_fwd_chunked_body(ex, a); } };
struct HeadBwdChunkBody { static MMX_D void run(Exec& ex, const ConvHeadBwdArgs& a) { conv_head_bwd_chunked_body(ex, a); } };
template <int WT>
struct HeadBwdBody { static MMX_D void run(Exec& ex, const ConvHeadBwdArgs& a) { conv_head_bwd_body<WT>(ex, a); } };

int check_enc(const MmxEncoderDesc* d, const MmxEncoderParams* w, const char* what) {
    if (!d || !w) return fail(MMX_E_INVALID, "%s: null descriptor / parameter table", what);
    if (d->B <= 0 || d->T <= 0 || d->D <= 0 || d->E <= 0 || d->C <= 0) return fail(MMX_E_INVALID, "%s: non-positive dimension", what);
    if (d->C > 8) return fail(MMX_E_UNSUPPORTED, "%s: conv_nChan %d > 8", what, d->C);
    if (!w->w || !w->b || !w->wc || !w->bc) return fail(MMX_E_INVALID, "%s: null parameter pointer", what);
    if (d->n_harmonic > 0 && !w->freq) return fail(MMX_E_INVALID, "%s: n_harmonic > 0 but frequencies is null", what);
    if ((d->E + 3) / 4 > kThreads) return fail(MMX_E_UNSUPPORTED, "%s: dimPosEmb %d too large", what, d->E);
    return MMX_OK;
}

constexpr int kEncChunkCols = 256;     // harmonic PoseEncoder forward: embedding columns (sin and cos) per chunk of input dimensions
constexpr int kEncBwdRows = 128;       // harmonic PoseEncoder backward, stage 2: frames staged per step of its sweep over the batch

// PoseEncoder forward.  A harmonic chunk is normally DC whole input dimensions (all Hn harmonics of each); when E rows of such
// a weight chunk do not fit shared memory, a chunk is one input dimension and HC of its harmonics (the widest HC that fits).
int plan_enc_fwd(const MmxEncoderDesc* d, EncDims* out, size_t* smem, int* grid) {
    const DevInfo di = dev_info();
    EncDims e;
    e.B = d->B; e.T = d->T; e.D = d->D; e.E = d->E; e.C = d->C; e.Hn = d->n_harmonic > 0 ? d->n_harmonic : 0;
    e.K = e.Hn > 0 ? 2 * e.Hn * e.D : e.D;
    const int rows = e.B * e.T, n_ct = (e.E + 3) / 4;
    auto fit = [&]() {
        int R = 64;
        while (R > 4 && ((R + 3) / 4) * n_ct > kThreads) R /= 2;
        while (R > 8 && (rows + R - 1) / R < di.sms) R /= 2;
        for (; R >= 4; R /= 2) {
            e.R = R;
            const size_t bytes = (size_t)enc_smem(e).total * 4;
            if (bytes <= (size_t)di.max_smem && ((R + 3) / 4) * n_ct <= kThreads) {
                *out = e; *smem = bytes; *grid = balanced_grid((rows + R - 1) / R, di.sms * ctas_per_sm(di, bytes, 8));
                return true;
            }
        }
        return false;
    };
    if (e.Hn == 0) {
        e.DC = 0; e.HC = 0;
        e.KC = imin(round_up(e.D, 4), 128);
        if (fit()) return MMX_OK;
    } else {
        const int forced_hc = env_int("MMX_ENC_HC", 0);   // tests: force the split chunk with this many harmonics
        if (forced_hc <= 0) {   // a chunk = DC input dimensions: their sin and cos columns (2*DC*Hn embedding columns)
            e.DC = imax(1, imin(e.D, kEncChunkCols / (2 * e.Hn)));
            e.HC = e.Hn;
            e.KC = round_up(2 * e.DC * e.Hn, 4);
            if (fit()) return MMX_OK;
        }
        for (int hc = forced_hc > 0 ? imin(forced_hc, e.Hn) : e.Hn; hc >= 1; hc /= 2) {
            e.DC = 1; e.HC = hc; e.KC = round_up(2 * hc, 4);
            if (fit()) return MMX_OK;
            if (forced_hc > 0) break;
        }
    }
    return fail(MMX_E_UNSUPPORTED, "PoseEncoder tile does not fit shared memory (D=%d E=%d)", d->D, d->E);
}

int check_head(const MmxConvHeadDesc* d, const MmxConvHeadParams* p, const char* what) {
    if (!d || !p) return fail(MMX_E_INVALID, "%s: null descriptor / parameter table", what);
    if (d->B <= 0 || d->C <= 0 || d->T <= 0 || d->To <= 0 || d->E <= 0 || d->D <= 0) return fail(MMX_E_INVALID, "%s: non-positive dimension", what);
    if (d->C > 8) return fail(MMX_E_UNSUPPORTED, "%s: conv_nChan %d > 8", what, d->C);
    if (!p->ln_w || !p->ln_b || !p->wt || !p->bt || !p->wp || !p->bp || !p->wf || !p->bf) return fail(MMX_E_INVALID, "%s: null parameter pointer", what);
    if (((d->To + 3) / 4) * ((d->T + 3) / 4) > kThreads) return fail(MMX_E_UNSUPPORTED, "%s: out_nTP %d too large", what, d->To);
    return MMX_OK;
}

// Resident plan (all of Wf in shared memory) when a tile fits; otherwise the chunked plan with the widest chunk that fits.
int plan_head(const MmxConvHeadDesc* d, bool bwd, ConvHeadDims* out, size_t* smem, int* grid) {
    const DevInfo di = dev_info();
    ConvHeadDims h; h.B = d->B; h.C = d->C; h.T = d->T; h.To = d->To; h.E = d->E; h.D = d->D; h.EC = 0;
    const int forced = env_int(bwd ? "MMX_CHEAD_S_BWD" : "MMX_CHEAD_S_FWD", 0);   // tests: force the tile
    const int forced_ec = env_int("MMX_CHEAD_EC", 0);                              // tests: force the chunked plan and its chunk
    auto start = [&](int width) {
        const int S0 = imax(1, 8192 / (imax(d->C * d->T, d->To) * width));
        return forced > 0 ? forced : imax(1, imin(S0, (d->B + 2 * di.sms - 1) / (2 * di.sms)));
    };
    auto take = [&](size_t bytes) {
        *out = h; *smem = bytes; *grid = tile_grid(di, d->B, h.S, bytes);
        return MMX_OK;
    };
    if (forced_ec <= 0) {
        const int S = fit_tile(di, start(d->E), forced > 0 ? forced : 1, 1, true, [&](int s) { h.S = s; return (size_t)conv_head_smem(h, bwd).total * 4; });
        if (S) { h.S = imin(S, d->B); return take((size_t)conv_head_smem(h, bwd).total * 4); }
    }
    for (int ec = forced_ec > 0 ? round_up(forced_ec, 4) : 128; ec >= (forced_ec > 0 ? 4 : 16); ec /= 2) {
        h.EC = ec;
        const int S = fit_tile(di, start(ec), forced > 0 ? forced : 1, 1, true, [&](int s) { h.S = s; return (size_t)conv_head_chunk_smem(h, bwd).total * 4; });
        if (S) { h.S = imin(S, d->B); return take((size_t)conv_head_chunk_smem(h, bwd).total * 4); }
        if (forced_ec > 0) break;
    }
    return fail(MMX_E_UNSUPPORTED, "ConvMixer head tile does not fit shared memory (C=%d E=%d D=%d To=%d)", d->C, d->E, d->D, d->To);
}

ConvHeadW to_hw(const MmxConvHeadParams* p) {
    ConvHeadW w; w.ln_g = p->ln_w; w.ln_b = p->ln_b; w.wt = p->wt; w.bt = p->bt; w.wp = p->wp; w.bp = p->bp; w.wf = p->wf; w.bf = p->bf;
    return w;
}
}  // namespace mmx_tu_conv_io
using namespace mmx_tu_conv_io;

extern "C" int mmx_linear_bwd(int rows, int K, int N, const float* x, const float* w, const float* dy, float* dw, float* db,
                              float* dx, void* stream);

extern "C" int mmx_pose_encoder_fwd(const MmxEncoderDesc* d, const MmxEncoderParams* w, const float* x, float* m, float* y, void* stream) {
    int rc = check_enc(d, w, "mmx_pose_encoder_fwd");
    if (rc) return rc;
    if (!x || !m || !y) return fail(MMX_E_INVALID, "mmx_pose_encoder_fwd: null tensor");
    EncFwdArgs a; size_t smem; int grid;
    if ((rc = plan_enc_fwd(d, &a.d, &smem, &grid))) return rc;
    a.w.freq = w->freq; a.w.w = w->w; a.w.b = w->b; a.w.wc = w->wc; a.w.bc = w->bc;
    a.x = x; a.m = m; a.y = y;
    return launch<EncFwdBody>(a, grid, kThreads, smem, stream);
}

extern "C" int mmx_pose_encoder_bwd(const MmxEncoderDesc* d, const MmxEncoderParams* w, const MmxEncoderParams* grads,
                                    const float* x, const float* m, const float* dy, float* dm_ws, float* dx, void* stream) {
    int rc = check_enc(d, w, "mmx_pose_encoder_bwd");
    if (rc) return rc;
    if (!grads || !grads->w || !grads->b || !grads->wc || !grads->bc) return fail(MMX_E_INVALID, "mmx_pose_encoder_bwd: null gradient pointer");
    if (!x || !m || !dy || !dm_ws) return fail(MMX_E_INVALID, "mmx_pose_encoder_bwd: null tensor");
    const DevInfo di = dev_info();
    const int rows = d->B * d->T, Hn = d->n_harmonic > 0 ? d->n_harmonic : 0;
    {
        EncBwd1Args a;
        a.d.B = d->B; a.d.T = d->T; a.d.E = d->E; a.d.C = d->C; a.d.R = 32; a.d.with_db = Hn > 0;
        a.wc = w->wc; a.m = m; a.dy = dy; a.dm = dm_ws; a.g_wc = grads->wc; a.g_bc = grads->bc; a.g_b = grads->b;
        const size_t smem = (size_t)enc_bwd1_smem(a.d).total * 4;
        if (smem > (size_t)di.max_smem) return fail(MMX_E_UNSUPPORTED, "mmx_pose_encoder_bwd: dimPosEmb %d too large", d->E);
        if ((rc = launch<EncBwd1Body>(a, balanced_grid((rows + 31) / 32, di.sms * 4), kThreads, smem, stream))) return rc;
    }
    if (Hn == 0) return mmx_linear_bwd(rows, d->D, d->E, x, w->w, dm_ws, grads->w, grads->b, dx, stream);
    EncBwd2Args a;
    a.d.B = d->B; a.d.T = d->T; a.d.D = d->D; a.d.E = d->E; a.d.Hn = Hn; a.d.need_dx = dx != nullptr;
    int HC = 32;
    while (HC > 2 && (HC > Hn || ((d->E + 3) / 4) * (2 * HC / 4) > kThreads)) HC /= 2;
    if (((d->E + 3) / 4) * (2 * HC / 4) > kThreads) return fail(MMX_E_UNSUPPORTED, "mmx_pose_encoder_bwd: dimPosEmb %d too large", d->E);
    a.d.HC = HC;
    a.freq = w->freq; a.w = w->w; a.x = x; a.dm = dm_ws; a.g_w = grads->w; a.dx = dx;
    // staged frames: kEncBwdRows, halved until the E-wide rows of dm fit shared memory
    const int forced_rows = env_int("MMX_ENC_BWD_ROWS", 0);   // tests: force the staged row count
    a.d.R = forced_rows > 0 ? forced_rows : kEncBwdRows;
    while (forced_rows <= 0 && a.d.R > 1 && (size_t)enc_bwd2_smem(a.d).total * 4 > (size_t)di.max_smem) a.d.R /= 2;
    const size_t smem = (size_t)enc_bwd2_smem(a.d).total * 4;
    if (smem > (size_t)di.max_smem) return fail(MMX_E_UNSUPPORTED, "mmx_pose_encoder_bwd: tile does not fit shared memory");
    if (dx && (rc = zero_async(dx, (size_t)rows * d->D * sizeof(float), stream))) return rc;
    const int groups = d->D * ((Hn + HC - 1) / HC);
    return launch<EncBwd2Body>(a, imin(groups, di.sms * 2), kThreads, smem, stream);
}

extern "C" int mmx_conv_head_fwd(const MmxConvHeadDesc* d, const MmxConvHeadParams* w, const float* y, float* out, void* stream) {
    int rc = check_head(d, w, "mmx_conv_head_fwd");
    if (rc) return rc;
    if (!y || !out) return fail(MMX_E_INVALID, "mmx_conv_head_fwd: null tensor");
    ConvHeadFwdArgs a; size_t smem; int grid;
    if ((rc = plan_head(d, false, &a.d, &smem, &grid))) return rc;
    a.w = to_hw(w); a.y = y; a.out = out;
    if (a.d.EC) return launch<HeadFwdChunkBody>(a, grid, kThreads, smem, stream);
    return launch<HeadFwdBody>(a, grid, kThreads, smem, stream);
}

extern "C" int mmx_conv_head_bwd(const MmxConvHeadDesc* d, const MmxConvHeadParams* w, const MmxConvHeadParams* grads,
                                 const float* y, const float* dout, float* dy, void* stream) {
    int rc = check_head(d, w, "mmx_conv_head_bwd");
    if (rc) return rc;
    if ((rc = check_head(d, grads, "mmx_conv_head_bwd(grads)"))) return rc;
    if (!y || !dout || !dy) return fail(MMX_E_INVALID, "mmx_conv_head_bwd: null tensor");
    ConvHeadBwdArgs a; size_t smem; int grid;
    if ((rc = plan_head(d, true, &a.d, &smem, &grid))) return rc;
    a.w = to_hw(w); a.g = to_hw(grads); a.y = y; a.dout = dout; a.dy = dy;
    if (a.d.EC) return launch<HeadBwdChunkBody>(a, grid, kThreads, smem, stream);
    const int tiles = ((d->D + 3) / 4) * ((d->E + 3) / 4);
    if (tiles <= kThreads) return launch<HeadBwdBody<1>>(a, grid, kThreads, smem, stream);
    return launch<HeadBwdBody<4>>(a, grid, kThreads, smem, stream);
}
