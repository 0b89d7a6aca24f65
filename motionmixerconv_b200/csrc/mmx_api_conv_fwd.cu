// mmx_conv_half_fwd, mmx_se_tail_{fwd,bwd} (include/mmx.h).
#include "mmx_conv_host.cuh"
#include "mmx_conv_io.cuh"

using namespace mmx;

namespace mmx_tu_conv_fwd {
template <int ACT, int CP>
struct ConvFwdBody { static MMX_D void run(Exec& ex, const ConvHalfFwdArgs& a) { conv_half_fwd_body<ACT, CP>(ex, a); } };
template <int ACT>
struct BnApplyBody { static MMX_D void run(Exec& ex, const BnPassArgs& a) { bn_apply_fwd_body<ACT>(ex, a); } };
template <int ACT>
struct BnBwd1Body { static MMX_D void run(Exec& ex, const BnPassArgs& a) { bn_bwd1_body<ACT>(ex, a); } };
struct SeTailFwdBody { static MMX_D void run(Exec& ex, const SeTailArgs& a) { se_tail_fwd_body(ex, a); } };
struct SeTailBwdBody { static MMX_D void run(Exec& ex, const SeTailArgs& a) { se_tail_bwd_body(ex, a); } };

template <int ACT>
int dispatch(const ConvHalfFwdArgs& a, int grid, size_t smem, void* stream) {
    switch (conv_cp(a.d.C)) {
        case 1: return launch<ConvFwdBody<ACT, 1>>(a, grid, kThreads, smem, stream);
        case 2: return launch<ConvFwdBody<ACT, 2>>(a, grid, kThreads, smem, stream);
        case 4: return launch<ConvFwdBody<ACT, 4>>(a, grid, kThreads, smem, stream);
        default: return launch<ConvFwdBody<ACT, 8>>(a, grid, kThreads, smem, stream);
    }
}

int plan_se_tail(int B, int C, int T, int E, int se_hidden, int use_se, int use_max, SeTailDims* out, size_t* smem, int* grid) {
    if (B <= 0 || C <= 0 || T <= 0 || E <= 0) return fail(MMX_E_INVALID, "non-positive dimension");
    if (T > 32) return fail(MMX_E_UNSUPPORTED, "in_nTP %d > 32", T);
    if (use_se && se_hidden < 1) return fail(MMX_E_UNSUPPORTED, "in_nTP // r_se == 0: empty SE bottleneck");
    SeTailDims d; d.B = B; d.C = C; d.T = T; d.E = E; d.rr = use_se ? se_hidden : 0; d.use_se = use_se; d.use_max = use_max;
    d.S = imin(B, imax(1, kConvTileElems / (C * T * E)));
    const DevInfo di = dev_info();
    *out = d; *smem = (size_t)se_tail_smem(d).total * 4;
    *grid = balanced_grid((B + d.S - 1) / d.S, di.sms * 4);
    return MMX_OK;
}
int plan_bn_pass(const MmxConvHalfDesc* d, BnPassDims* out, size_t* smem, int* grid) {
    if (!d) return fail(MMX_E_INVALID, "null descriptor");
    if (d->B <= 0 || d->C <= 0 || d->T <= 0 || d->E <= 0) return fail(MMX_E_INVALID, "non-positive dimension");
    if (d->C > 8 || d->T > 32) return fail(MMX_E_UNSUPPORTED, "conv_nChan %d > 8 or in_nTP %d > 32", d->C, d->T);
    if (d->act != MMX_ACT_GELU && d->act != MMX_ACT_MISH) return fail(MMX_E_INVALID, "Unknown activation function type: %d", d->act);
    if (d->use_se && d->se_hidden < 1) return fail(MMX_E_UNSUPPORTED, "in_nTP // r_se == 0: empty SE bottleneck");
    if (d->use_se && d->use_max_pooling) return fail(MMX_E_UNSUPPORTED, "BatchNorm halves support the mean squeeze only");
    BnPassDims b; b.B = d->B; b.C = d->C; b.T = d->T; b.E = d->E; b.rr = d->use_se ? d->se_hidden : 0; b.use_se = d->use_se; b.act = d->act;
    b.S = imin(d->B, imax(1, kConvTileElems / (d->C * d->T * d->E)));
    const DevInfo di = dev_info();
    *out = b; *smem = (size_t)bn_pass_smem(b).total * 4;
    *grid = balanced_grid((d->B + b.S - 1) / b.S, di.sms * 4);
    return MMX_OK;
}
}  // namespace mmx_tu_conv_fwd
using namespace mmx_tu_conv_fwd;

extern "C" int mmx_conv_half_bn_stats(const MmxConvHalfDesc* d, const MmxConvHalfParams* w, const float* x, float* z, double* sums, void* stream) {
    if (!x || !z || !sums) return fail(MMX_E_INVALID, "mmx_conv_half_bn_stats: null tensor");
    ConvHalfFwdArgs a;
    size_t smem; int grid;
    int rc = plan_conv_half(d, false, &a.d, &smem, &grid);
    if (rc) return rc;
    if ((rc = check_conv_params(w, 0, "mmx_conv_half_bn_stats"))) return rc;
    a.d.bn_mode = 1; a.d.use_se = 0; a.d.rr = 0; a.d.training = 0;      // statistics pass: LN -> conv -> act only
    a.dr = make_dropout(d->dropout, 0);
    a.w = to_cw(w); a.x = x; a.y = nullptr; a.aff = nullptr; a.zout = z; a.bnsum = sums;
    return d->act == MMX_ACT_GELU ? dispatch<ACT_GELU>(a, grid, smem, stream) : dispatch<ACT_MISH>(a, grid, smem, stream);
}

extern "C" int mmx_conv_half_bn_apply(const MmxConvHalfDesc* d, const MmxConvHalfParams* w, const float* bn, const float* x,
                                      const float* z, float* y, void* stream) {
    if (!bn || !x || !z || !y) return fail(MMX_E_INVALID, "mmx_conv_half_bn_apply: null tensor");
    BnPassArgs a; size_t smem; int grid;
    int rc = plan_bn_pass(d, &a.d, &smem, &grid);
    if (rc) return rc;
    if (d->use_se && (!w || !w->se_w1 || !w->se_w2)) return fail(MMX_E_INVALID, "mmx_conv_half_bn_apply: use_se set but SE weights are null");
    a.se1 = w ? w->se_w1 : nullptr; a.se2 = w ? w->se_w2 : nullptr; a.g_se1 = a.g_se2 = nullptr;
    a.bn = bn; a.x = x; a.z = z; a.dy = nullptr; a.y = y; a.gd = nullptr; a.sums = nullptr;
    return d->act == MMX_ACT_GELU ? launch<BnApplyBody<ACT_GELU>>(a, grid, kThreads, smem, stream)
                                  : launch<BnApplyBody<ACT_MISH>>(a, grid, kThreads, smem, stream);
}

extern "C" int mmx_conv_half_bn_bwd1(const MmxConvHalfDesc* d, const MmxConvHalfParams* w, const MmxConvHalfParams* grads, const float* bn,
                                     const float* z, const float* dy, float* gd, double* sums, void* stream) {
    if (!bn || !z || !dy || !gd || !sums) return fail(MMX_E_INVALID, "mmx_conv_half_bn_bwd1: null tensor");
    BnPassArgs a; size_t smem; int grid;
    int rc = plan_bn_pass(d, &a.d, &smem, &grid);
    if (rc) return rc;
    if (d->use_se && (!w || !w->se_w1 || !w->se_w2 || !grads || !grads->se_w1 || !grads->se_w2))
        return fail(MMX_E_INVALID, "mmx_conv_half_bn_bwd1: use_se set but SE weights / grads are null");
    a.se1 = w ? w->se_w1 : nullptr; a.se2 = w ? w->se_w2 : nullptr;
    a.g_se1 = grads ? grads->se_w1 : nullptr; a.g_se2 = grads ? grads->se_w2 : nullptr;
    a.bn = bn; a.x = nullptr; a.z = z; a.dy = dy; a.y = nullptr; a.gd = gd; a.sums = sums;
    return d->act == MMX_ACT_GELU ? launch<BnBwd1Body<ACT_GELU>>(a, grid, kThreads, smem, stream)
                                  : launch<BnBwd1Body<ACT_MISH>>(a, grid, kThreads, smem, stream);
}

extern "C" int mmx_conv_half_fwd(const MmxConvHalfDesc* d, const MmxConvHalfParams* w, const float* x, float* y, void* stream) {
    if (!x || !y) return fail(MMX_E_INVALID, "mmx_conv_half_fwd: null tensor");
    ConvHalfFwdArgs a;
    size_t smem; int grid;
    int rc = plan_conv_half(d, false, &a.d, &smem, &grid);
    if (rc) return rc;
    if ((rc = check_conv_params(w, d->use_se, "mmx_conv_half_fwd"))) return rc;
    a.dr = make_dropout(d->dropout, d->training);
    a.w = to_cw(w); a.x = x; a.y = y; a.aff = w->bn_aff; a.zout = nullptr; a.bnsum = nullptr;
    return d->act == MMX_ACT_GELU ? dispatch<ACT_GELU>(a, grid, smem, stream) : dispatch<ACT_MISH>(a, grid, smem, stream);
}

// capability query: does the fused half kernel serve this descriptor (forward / backward)?  MMX_OK + the plan, or the error the
// compute entry point would return.  No launch; the ConvMixer module uses it to report unsupported shapes at construction.
extern "C" int mmx_conv_half_plan(const MmxConvHalfDesc* d, int backward, int* seq_per_tile, int* smem_bytes) {
    ConvDims m; size_t smem; int grid;
    int rc = plan_conv_half(d, backward != 0, &m, &smem, &grid);
    if (rc) return rc;
    if (seq_per_tile) *seq_per_tile = m.S;
    if (smem_bytes) *smem_bytes = (int)smem;
    return MMX_OK;
}

extern "C" int mmx_se_tail_fwd(int B, int C, int T, int E, int se_hidden, int use_se, int use_max_pooling,
                               const float* se_w1, const float* se_w2, const float* x, float* y, void* stream) {
    if (!x || !y) return fail(MMX_E_INVALID, "mmx_se_tail_fwd: null tensor");
    if (use_se && (!se_w1 || !se_w2)) return fail(MMX_E_INVALID, "mmx_se_tail_fwd: use_se set but SE weights are null");
    SeTailArgs a; size_t smem; int grid;
    int rc = plan_se_tail(B, C, T, E, se_hidden, use_se, use_max_pooling, &a.d, &smem, &grid);
    if (rc) return rc;
    a.se1 = se_w1; a.se2 = se_w2; a.g_se1 = a.g_se2 = nullptr; a.x = x; a.dy = nullptr; a.out = y;
    return launch<SeTailFwdBody>(a, grid, kThreads, smem, stream);
}

extern "C" int mmx_se_tail_bwd(int B, int C, int T, int E, int se_hidden, int use_se, int use_max_pooling,
                               const float* se_w1, const float* se_w2, float* g_se_w1, float* g_se_w2,
                               const float* x, const float* dy, float* dx, void* stream) {
    if (!x || !dy || !dx) return fail(MMX_E_INVALID, "mmx_se_tail_bwd: null tensor");
    if (use_se && (!se_w1 || !se_w2 || !g_se_w1 || !g_se_w2)) return fail(MMX_E_INVALID, "mmx_se_tail_bwd: use_se set but SE weights / grads are null");
    SeTailArgs a; size_t smem; int grid;
    int rc = plan_se_tail(B, C, T, E, se_hidden, use_se, use_max_pooling, &a.d, &smem, &grid);
    if (rc) return rc;
    a.se1 = se_w1; a.se2 = se_w2; a.g_se1 = g_se_w1; a.g_se2 = g_se_w2; a.x = x; a.dy = dy; a.out = dx;
    return launch<SeTailBwdBody>(a, grid, kThreads, smem, stream);
}
