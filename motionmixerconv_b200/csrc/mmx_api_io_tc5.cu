// Embedding (per-frame Linear) and output head of the MlpMixer on the Blackwell tensor cores: launch layer of
// mmx_lin_tc5.cuh and mmx_head_tc5.cuh.  Reached from mmx_linear_{fwd,bwd}_prec / mmx_mlp_head_{fwd,bwd}_prec when the caller
// asks for the reduced-precision mode (MMX_PREC_TF32) and the shape is served; everything else stays on the fp32 kernels.
#include "mmx_launch.cuh"

#if defined(MMX_HOST_EMU)
bool mmx_lin_tc5_ok(long long, int, int, const void*, const void*, const void*) { return false; }
int mmx_lin_tc5(bool, long long, int, int, const float*, const float*, const float*, const float*, float*, float*, float*, void*) {
    return fail(MMX_E_UNSUPPORTED, "no tensor cores in the emulator");
}
bool mmx_head_tc5_ok(const MmxMlpHeadDesc*) { return false; }
int mmx_head_tc5(bool, const MmxMlpHeadDesc*, const MmxMlpHeadParams*, const MmxMlpHeadParams*, const float*, const float*, float*, void*) {
    return fail(MMX_E_UNSUPPORTED, "no tensor cores in the emulator");
}
#else
#include "mmx_head_tc5.cuh"
#include "mmx_lin_tc5.cuh"

using namespace mmx;

// ------------------------------------------------------------------------------------------ linear layer on rows
bool mmx_lin_tc5_ok(long long rows, int K, int N, const void* x, const void* y, const void* dx) {
    if (env_int("MMX_IO_NO_TC5", 0)) return false;
    if (rows <= 0 || K < 8 || N < 8 || (K & 1) || (N & 1)) return false;
    if (K + 1 > 80 || N > 80) return false;                          // one padded operand width serves both sides (+ the ones column)
    if (((rows * K) & 3) || ((rows * N) & 3)) return false;          // bulk copies: every tile is a multiple of 16 bytes
    if ((((uintptr_t)x) | ((uintptr_t)y) | ((uintptr_t)dx)) & 15) return false;
    return true;
}

// forward: out = y = x W^T + b (dy, dw, db unused); backward: dw += dY^T x, db += column sums of dY, out = dx (nullable)
int mmx_lin_tc5(bool bwd, long long rows, int K, int N, const float* x, const float* w, const float* b, const float* dy, float* dw,
                float* db, float* out, void* stream) {
    lin::LinArgs a;
    a.x = x; a.w = w; a.b = b; a.dy = dy; a.out = out; a.g_w = dw; a.g_b = db;
    a.R = rows; a.K = K; a.N = N;
    a.abort_count = mmx_tc5_abort_ptr();
    const DevInfo di = dev_info();
    const bool small = (K + 1 > N ? K + 1 : N) <= 64;
    const size_t smem = small ? lin::lin_smem<64>(K, N, bwd).total : lin::lin_smem<80>(K, N, bwd).total;
    const int grid = capped_grid(di, rows, 128, ctas_per_sm(di, smem, 2));        // rows >= 1: mmx_lin_tc5_ok
    const auto kern = bwd ? (small ? lin::lin_bwd_kernel<64, 2> : lin::lin_bwd_kernel<80, 2>)
                          : (small ? lin::lin_fwd_kernel<64, 2> : lin::lin_fwd_kernel<80, 2>);
    return launch_kernel(kern, grid, tc5::kCtaThreads, smem, stream, kPdl, a);
}

// ------------------------------------------------------------------------------------------ output head
bool mmx_head_tc5_ok(const MmxMlpHeadDesc* d) {
    if (env_int("MMX_IO_NO_TC5", 0)) return false;
    if (d->B <= 0 || d->T < 1 || d->To < 1 || d->T > 128 || d->To > 128) return false;
    if (d->H < 8 || d->D < 8 || (d->H & 1) || (d->D & 1) || d->H + 1 > head::KH || d->D > head::KD) return false;
    if (((d->T * d->H) & 3) || ((d->To * d->D) & 3)) return false;
    return true;
}

// forward: out = head(x) (grads, dout unused); backward: grads += parameter gradients, out = dx
int mmx_head_tc5(bool bwd, const MmxMlpHeadDesc* d, const MmxMlpHeadParams* w, const MmxMlpHeadParams* grads, const float* x,
                 const float* dout, float* out, void* stream) {
    head::HeadArgs a;
    a.ln_g = w->ln_w; a.ln_b = w->ln_b; a.wt = w->wt; a.bt = w->bt; a.wf = w->wf; a.bf = w->bf;
    if (bwd) { a.g_ln_g = grads->ln_w; a.g_ln_b = grads->ln_b; a.g_wt = grads->wt; a.g_bt = grads->bt; a.g_wf = grads->wf; a.g_bf = grads->bf; }
    else a.g_ln_g = a.g_ln_b = a.g_wt = a.g_bt = a.g_wf = a.g_bf = nullptr;
    a.B = d->B; a.T = d->T; a.To = d->To; a.H = d->H; a.D = d->D;
    a.S = 128 / imax(d->T, d->To);
    a.x = x; a.dout = bwd ? dout : nullptr; a.out = out;
    a.abort_count = mmx_tc5_abort_ptr();
    const int grid = capped_grid(dev_info(), d->B, a.S, 1);        // B >= 1 and S >= 1: mmx_head_tc5_ok
    const size_t smem = head::head_smem(d->H, d->D, bwd).total;
    return launch_kernel(bwd ? head::head_bwd_kernel : head::head_fwd_kernel, grid, tc5::kCtaThreads, smem, stream, kPdl, a);
}
#endif
