// mmx_window_split, mmx_pck_hist (include/mmx.h).
#include "mmx_launch.cuh"
#include "mmx_aux.cuh"

using namespace mmx;

namespace mmx_tu_aux {
struct WindowSplitBody { static MMX_D void run(Exec& ex, const WindowSplitArgs& a) { window_split_body(ex, a); } };
struct BnFinalizeBody { static MMX_D void run(Exec& ex, const BnFinalizeArgs& a) { bn_finalize_body(ex, a); } };
struct BnCoefBody { static MMX_D void run(Exec& ex, const BnCoefArgs& a) { bn_coef_body(ex, a); } };
struct PckHistBody { static MMX_D void run(Exec& ex, const PckHistArgs& a) { pck_hist_body(ex, a); } };
}  // namespace mmx_tu_aux
using namespace mmx_tu_aux;

extern "C" int mmx_window_split(const float* batch, int B, int Ttot, int Dfull, const int* dim_used, int D, int T, int To,
                                float x_scale, float gt_scale, float* x, float* gt, void* stream) {
    if (!batch || !dim_used || !x || !gt) return fail(MMX_E_INVALID, "mmx_window_split: null tensor");
    if (B <= 0 || D <= 0 || T <= 0 || To <= 0 || Dfull <= 0 || T + To > Ttot) return fail(MMX_E_INVALID, "mmx_window_split: bad window geometry");
    WindowSplitArgs a;
    a.batch = batch; a.dim_used = dim_used; a.x = x; a.gt = gt; a.B = B; a.Ttot = Ttot; a.Dfull = Dfull; a.D = D; a.T = T; a.To = To;
    a.x_scale = x_scale; a.gt_scale = gt_scale;
    return launch<WindowSplitBody>(a, capped_grid(dev_info(), (long long)B * (T + To) * D, kThreads * 4, 8), kThreads, 16, stream);
}

extern "C" int mmx_pck_hist(const float* pred, const float* gt, long long n_joints, const float* thresh, int n, int* hist, void* stream) {
    if (!pred || !gt || !thresh || !hist) return fail(MMX_E_INVALID, "mmx_pck_hist: null tensor");
    if (n_joints <= 0 || n <= 0 || n > 4096) return fail(MMX_E_INVALID, "mmx_pck_hist: bad sizes");
    PckHistArgs a; a.pred = pred; a.gt = gt; a.thresh = thresh; a.hist = hist; a.n_joints = n_joints; a.n = n;
    return launch<PckHistBody>(a, capped_grid(dev_info(), n_joints, kThreads * 4, 4), kThreads, (size_t)(2 * n + 8) * 4, stream);
}

extern "C" int mmx_bn_finalize(double* sums, int C, double n, const float* w, const float* b, float* running_mean, float* running_var,
                               long long* num_batches_tracked, float momentum, float eps, float* bn, void* stream) {
    if (!sums || !w || !b || !running_mean || !running_var || !num_batches_tracked || !bn) return fail(MMX_E_INVALID, "mmx_bn_finalize: null tensor");
    if (C <= 0 || !(n >= 1.0)) return fail(MMX_E_INVALID, "mmx_bn_finalize: bad sizes");
    BnFinalizeArgs a; a.sums = sums; a.w = w; a.b = b; a.rm = running_mean; a.rv = running_var; a.nbt = num_batches_tracked; a.bn = bn;
    a.n = n; a.momentum = momentum; a.eps = eps; a.C = C;
    return launch<BnFinalizeBody>(a, (C + 31) / 32, 32, 16, stream);
}

extern "C" int mmx_bn_coef(double* sums, int C, double n, const float* bn, float* coef, float* g_weight, float* g_bias, void* stream) {
    if (!sums || !bn || !coef || !g_weight || !g_bias) return fail(MMX_E_INVALID, "mmx_bn_coef: null tensor");
    if (C <= 0 || !(n >= 1.0)) return fail(MMX_E_INVALID, "mmx_bn_coef: bad sizes");
    BnCoefArgs a; a.sums = sums; a.bn = bn; a.coef = coef; a.gw = g_weight; a.gb = g_bias; a.n = n; a.C = C;
    return launch<BnCoefBody>(a, (C + 31) / 32, 32, 16, stream);
}
