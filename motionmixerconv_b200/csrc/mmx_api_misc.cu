// Entry points: linear (embedding), MlpMixer head, MPJPE, Adam, version / error reporting.
#include <string>

#include "mmx_launch.cuh"
#include "mmx_loss_adam.cuh"
#include "mmx_mlp.cuh"

using namespace mmx;

static thread_local std::string g_err;
#undef fail
int mmx_fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
#define fail mmx_fail

namespace mmx_tu_misc {
// ---------------------------------------------------------------------------------- linear / head / loss / adam
struct LinFwdBody { static MMX_D void run(Exec& ex, const LinearFwdArgs& a) { linear_fwd_body(ex, a); } };
template <int WT>
struct LinBwdBody { static MMX_D void run(Exec& ex, const LinearBwdArgs& a) { linear_bwd_body<WT>(ex, a); } };
template <int TC>
struct HeadFwdBody { static MMX_D void run(Exec& ex, const MlpHeadFwdArgs& a) { mlp_head_fwd_body<TC>(ex, a); } };
template <int TC, int WT>
struct HeadBwdBody { static MMX_D void run(Exec& ex, const MlpHeadBwdArgs& a) { mlp_head_bwd_body<TC, WT>(ex, a); } };
struct MpjpeBody { static MMX_D void run(Exec& ex, const MpjpeArgs& a) { mpjpe_body(ex, a); } };
struct AdamBody { static MMX_D void run(Exec& ex, const AdamArgs& a) { adam_body(ex, a); } };
struct AdamAdvanceBody { static MMX_D void run(Exec& ex, const AdamAdvanceArgs& a) { adam_advance_body(ex, a); } };

int plan_linear(int rows, int K, int N, bool bwd, LinearDims* out, size_t* smem, int* grid) {
    if (rows <= 0 || K <= 0 || N <= 0) return fail(MMX_E_INVALID, "non-positive dimension");
    const DevInfo di = dev_info();
    LinearDims d; d.rows = rows; d.K = K; d.N = N;
    const int R = fit_tile(di, 128, 8, 8, true, [&](int r) { d.R = r; return (size_t)linear_smem(d, bwd).total * 4; });
    if (!R) return fail(MMX_E_UNSUPPORTED, "linear layer K=%d N=%d does not fit shared memory", K, N);
    d.R = imin(R, round_up(rows, 4));
    if (d.R == R && R >= 16) d.R = balanced_tile(rows, R, R / 2, 8, di.sms);
    const size_t bytes = (size_t)linear_smem(d, bwd).total * 4;
    *out = d; *smem = bytes; *grid = tile_grid(di, rows, d.R, bytes);
    return MMX_OK;
}

int check_head_desc(const MmxMlpHeadDesc* d) {
    if (!d) return fail(MMX_E_INVALID, "null descriptor");
    if (d->B <= 0 || d->T <= 0 || d->To <= 0 || d->H <= 0 || d->D <= 0) return fail(MMX_E_INVALID, "non-positive dimension");
    return MMX_OK;
}

int plan_head(const MmxMlpHeadDesc* d, bool bwd, MlpHeadDims* out, size_t* smem, int* grid) {
    if (int rc = check_head_desc(d)) return rc;
    if (d->T > 32) return fail(MMX_E_UNSUPPORTED, "seq_len %d > 32", d->T);
    if (((d->To + 3) / 4) * ((d->T + 3) / 4) > kThreads) return fail(MMX_E_UNSUPPORTED, "pred_len %d too large", d->To);
    const DevInfo di = dev_info();
    MlpHeadDims h; h.B = d->B; h.T = d->T; h.To = d->To; h.H = d->H; h.D = d->D;
    // sequences per tile: ~96 output rows per tile for narrow models.  Wide rows (H >= 64: K4, H = 128) amortise the fc_out weight
    // reads over more rows, and one CTA per SM with a larger tile beats two CTAs with S = 2 -- measured in the one-CTA budget at
    // B = 4096, T = 10, To = 25, H = 128, D = 54 (us, fwd / bwd): S = 2: 122 / 400, 4: 98 / 302, 6: 120 / 285
    const int rows0 = d->H >= 64 ? (bwd ? 160 : 100) : 96;
    const int S = fit_tile(di, imax(1, rows0 / imax(d->T, d->To)), 1, 1, d->H < 64,
                           [&](int s) { h.S = s; return (size_t)mlp_head_smem(h, bwd).total * 4; });
    if (!S) return fail(MMX_E_UNSUPPORTED, "MlpMixer head tile does not fit shared memory (H=%d D=%d To=%d)", d->H, d->D, d->To);
    h.S = imin(S, d->B);
    if (h.S == S && S >= 2) h.S = balanced_tile(d->B, S, (S + 1) / 2, 1, di.sms);
    const size_t bytes = (size_t)mlp_head_smem(h, bwd).total * 4;
    *out = h; *smem = bytes; *grid = tile_grid(di, d->B, h.S, bytes);
    return MMX_OK;
}


}  // namespace mmx_tu_misc
using namespace mmx_tu_misc;

// tcgen05 kernels of the embedding / output head (mmx_api_io_tc5.cu)
bool mmx_lin_tc5_ok(long long rows, int K, int N, const void* x, const void* y, const void* dx);
int mmx_lin_tc5(bool bwd, long long rows, int K, int N, const float* x, const float* w, const float* b, const float* dy, float* dw,
                float* db, float* out, void* stream);
bool mmx_head_tc5_ok(const MmxMlpHeadDesc* d);
int mmx_head_tc5(bool bwd, const MmxMlpHeadDesc* d, const MmxMlpHeadParams* w, const MmxMlpHeadParams* grads, const float* x,
                 const float* dout, float* out, void* stream);

// ====================================================================================== C ABI
extern "C" {

int mmx_version(void) { return 100; }
const char* mmx_last_error(void) { return g_err.c_str(); }

int mmx_linear_fwd(int rows, int K, int N, const float* x, const float* w, const float* b, float* y, void* stream) {
    return mmx_linear_fwd_prec(rows, K, N, x, w, b, y, MMX_PREC_FP32, stream);
}
int mmx_linear_bwd(int rows, int K, int N, const float* x, const float* w, const float* dy, float* dw, float* db, float* dx, void* stream) {
    return mmx_linear_bwd_prec(rows, K, N, x, w, dy, dw, db, dx, MMX_PREC_FP32, stream);
}

int mmx_linear_fwd_prec(int rows, int K, int N, const float* x, const float* w, const float* b, float* y, int precision, void* stream) {
    if (!x || !w || !b || !y) return fail(MMX_E_INVALID, "mmx_linear_fwd: null tensor");
    if (precision == MMX_PREC_TF32 && mmx_lin_tc5_ok(rows, K, N, x, y, nullptr)) return mmx_lin_tc5(false, rows, K, N, x, w, b, nullptr, nullptr, nullptr, y, stream);
    LinearFwdArgs a; size_t smem; int grid;
    int rc = plan_linear(rows, K, N, false, &a.d, &smem, &grid);
    if (rc) return rc;
    a.x = x; a.w = w; a.b = b; a.y = y;
    return launch<LinFwdBody>(a, grid, kThreads, smem, stream);
}

int mmx_linear_bwd_prec(int rows, int K, int N, const float* x, const float* w, const float* dy, float* dw, float* db,
                        float* dx, int precision, void* stream) {
    if (!x || !w || !dy || !dw || !db) return fail(MMX_E_INVALID, "mmx_linear_bwd: null tensor");
    if (precision == MMX_PREC_TF32 && mmx_lin_tc5_ok(rows, K, N, x, dy, dx)) return mmx_lin_tc5(true, rows, K, N, x, w, nullptr, dy, dw, db, dx, stream);
    LinearBwdArgs a; size_t smem; int grid;
    int rc = plan_linear(rows, K, N, true, &a.d, &smem, &grid);
    if (rc) return rc;
    a.x = x; a.w = w; a.dy = dy; a.dw = dw; a.db = db; a.dx = dx;
    const int tiles = ((N + 3) / 4) * ((K + 3) / 4);
    if (tiles <= kThreads) return launch<LinBwdBody<1>>(a, grid, kThreads, smem, stream);
    return launch<LinBwdBody<4>>(a, grid, kThreads, smem, stream);
}

static MlpHeadW to_hw(const MmxMlpHeadParams* p) {
    MlpHeadW w; w.ln_g = p->ln_w; w.ln_b = p->ln_b; w.wt = p->wt; w.bt = p->bt; w.wf = p->wf; w.bf = p->bf; return w;
}
static int check_head_params(const MmxMlpHeadParams* p, const char* what) {
    if (!p || !p->ln_w || !p->ln_b || !p->wt || !p->bt || !p->wf || !p->bf) return fail(MMX_E_INVALID, "%s: null parameter pointer", what);
    return MMX_OK;
}

int mmx_mlp_head_fwd(const MmxMlpHeadDesc* d, const MmxMlpHeadParams* w, const float* x, float* out, void* stream) {
    return mmx_mlp_head_fwd_prec(d, w, x, out, MMX_PREC_FP32, stream);
}
int mmx_mlp_head_bwd(const MmxMlpHeadDesc* d, const MmxMlpHeadParams* w, const MmxMlpHeadParams* grads,
                     const float* x, const float* dout, float* dx, void* stream) {
    return mmx_mlp_head_bwd_prec(d, w, grads, x, dout, dx, MMX_PREC_FP32, stream);
}

int mmx_mlp_head_fwd_prec(const MmxMlpHeadDesc* d, const MmxMlpHeadParams* w, const float* x, float* out, int precision, void* stream) {
    if (!x || !out) return fail(MMX_E_INVALID, "mmx_mlp_head_fwd: null tensor");
    int rc = check_head_desc(d);
    if (rc) return rc;
    if ((rc = check_head_params(w, "mmx_mlp_head_fwd"))) return rc;
    // the tcgen05 head serves T, To <= 128; the fp32 planner below stops at T = 32, so it is asked only when tcgen05 declines
    if (precision == MMX_PREC_TF32 && mmx_head_tc5_ok(d) && !((((uintptr_t)x) | ((uintptr_t)out)) & 15)) return mmx_head_tc5(false, d, w, nullptr, x, nullptr, out, stream);
    MlpHeadFwdArgs a; size_t smem; int grid;
    if ((rc = plan_head(d, false, &a.d, &smem, &grid))) return rc;
    a.w = to_hw(w); a.x = x; a.out = out;
    if (d->T == 10) return launch<HeadFwdBody<10>>(a, grid, kThreads, smem, stream);
    return launch<HeadFwdBody<0>>(a, grid, kThreads, smem, stream);
}

int mmx_mlp_head_bwd_prec(const MmxMlpHeadDesc* d, const MmxMlpHeadParams* w, const MmxMlpHeadParams* grads,
                          const float* x, const float* dout, float* dx, int precision, void* stream) {
    if (!x || !dout || !dx) return fail(MMX_E_INVALID, "mmx_mlp_head_bwd: null tensor");
    int rc = check_head_desc(d);
    if (rc) return rc;
    if ((rc = check_head_params(w, "mmx_mlp_head_bwd"))) return rc;
    if ((rc = check_head_params(grads, "mmx_mlp_head_bwd(grads)"))) return rc;
    if (precision == MMX_PREC_TF32 && mmx_head_tc5_ok(d) && !((((uintptr_t)x) | ((uintptr_t)dout) | ((uintptr_t)dx)) & 15))
        return mmx_head_tc5(true, d, w, grads, x, dout, dx, stream);
    MlpHeadBwdArgs a; size_t smem; int grid;
    if ((rc = plan_head(d, true, &a.d, &smem, &grid))) return rc;
    a.w = to_hw(w); a.g = to_hw(grads); a.x = x; a.dout = dout; a.dx = dx;
    const int tiles = ((d->D + 3) / 4) * ((d->H + 3) / 4);
    if (d->T == 10) {
        if (tiles <= kThreads) return launch<HeadBwdBody<10, 1>>(a, grid, kThreads, smem, stream);
        return launch<HeadBwdBody<10, 4>>(a, grid, kThreads, smem, stream);
    }
    if (tiles <= kThreads) return launch<HeadBwdBody<0, 1>>(a, grid, kThreads, smem, stream);
    return launch<HeadBwdBody<0, 4>>(a, grid, kThreads, smem, stream);
}

int mmx_mpjpe_fwd_bwd(const float* pred, const float* gt, float* dpred, float* loss_sum, long long n_joints,
                      float gscale, void* stream) {
    if (!pred || !gt || !loss_sum) return fail(MMX_E_INVALID, "mmx_mpjpe_fwd_bwd: null tensor");
    if (n_joints <= 0) return fail(MMX_E_INVALID, "mmx_mpjpe_fwd_bwd: n_joints must be positive");
    MpjpeArgs a; a.pred = pred; a.gt = gt; a.dpred = dpred; a.loss_sum = loss_sum; a.n_joints = n_joints; a.gscale = gscale;
    return launch<MpjpeBody>(a, capped_grid(dev_info(), n_joints, kThreads, 8), kThreads, kThreads * sizeof(float), stream);
}

int mmx_adam_step(float* p, const float* g, float* m, float* v, long long n, const float* hyper, void* stream) {
    if (!p || !g || !m || !v || !hyper) return fail(MMX_E_INVALID, "mmx_adam_step: null tensor");
    if (n <= 0) return fail(MMX_E_INVALID, "mmx_adam_step: n must be positive");
    if ((((uintptr_t)p) | ((uintptr_t)g) | ((uintptr_t)m) | ((uintptr_t)v)) & 15) return fail(MMX_E_INVALID, "mmx_adam_step: buffers must be 16-byte aligned");
    AdamArgs a; a.p = p; a.g = g; a.m = m; a.v = v; a.hp = hyper; a.n = n;
    const DevInfo di = dev_info();
    const long long want = ((n >> 2) + kThreads - 1) / kThreads + 1;
    const int grid = (int)(want < (long long)di.sms * 8 ? want : (long long)di.sms * 8);
    return launch<AdamBody>(a, grid, kThreads, 16, stream);
}

int mmx_adam_advance(float* hyper, unsigned int* step, void* stream) {
    if (!hyper || !step) return fail(MMX_E_INVALID, "mmx_adam_advance: null pointer");
    AdamAdvanceArgs a; a.hp = hyper; a.step = step;
    return launch<AdamAdvanceBody>(a, 1, 32, 16, stream);
}

}  // extern "C"
