// The ConvBlock convolution of the stage-kernel chain in the reduced-precision mode: launch layer of mmx_conv_tc5.cuh and the
// precision-aware entry points mmx_conv2d_large_{fwd,wgrad}_prec.  MMX_PREC_TF32 runs the convolution on tcgen05 when
// mmx_conv2d_tc5_serves(d); every other call is the fp32 entry point (mmx_api_conv_large.cu), bit for bit.
#include "mmx_launch.cuh"

#if defined(MMX_HOST_EMU)
static bool conv_tc5_ok(const MmxConvHalfDesc*) { return false; }
static int conv_tc5_fwd(const MmxConvHalfDesc*, int, const float*, const float*, const float*, float*, void*) {
    return fail(MMX_E_UNSUPPORTED, "no tensor cores in the emulator");
}
static int conv_tc5_wgrad(const MmxConvHalfDesc*, const float*, const float*, float*, float*, void*) {
    return fail(MMX_E_UNSUPPORTED, "no tensor cores in the emulator");
}
#else
#include "mmx_conv_tc5.cuh"
#include "mmx_tc5_launch.cuh"

using namespace mmx;

static bool conv_tc5_ok(const MmxConvHalfDesc* d) {
    if (!d || d->B <= 0 || d->C < 1 || d->C > 8 || d->T < 1 || d->E < 1 || d->kt < 1 || d->kp < 1) return false;
    if (d->pad_t < 0 || d->pad_p < 0 || d->pad_t > d->kt - 1 || d->pad_p > d->kp - 1) return false;
    const ctc5::ConvGeom g = ctc5::conv_tc5_geom(d->C, d->T, d->E, d->kt, d->kp);
    if (g.NP > 256 || g.Kp > 128 || g.ST < 8) return false;      // MMA N <= 256; wgrad accumulators <= 2 x 128 TMEM columns
    const int smax = dev_info().max_smem;
    return (int)ctc5::conv_tc5_smem(g, d->C, false).total <= smax && (int)ctc5::conv_tc5_smem(g, d->C, true).total <= smax;
}

static ctc5::ConvTc5Args conv_args(const MmxConvHalfDesc* d) {
    ctc5::ConvTc5Args a = {};
    a.B = d->B; a.C = d->C; a.T = d->T; a.E = d->E; a.kt = d->kt; a.kp = d->kp; a.pt = d->pad_t; a.pp = d->pad_p;
    a.abort_count = mmx_tc5_abort_ptr();
    return a;
}

// CTAs: one per SM (the plans of the Optuna cells take most of shared memory); more where shared memory and TMEM allow
static int conv_grid(const ctc5::ConvGeom& g, int B, size_t smem, int tm_cols) {
    const DevInfo di = dev_info();
    const int per_sm = imax(1, imin(512 / tm_cols, (int)((di.max_smem + 1024) / (smem + 1024))));
    const long long items = (long long)B * g.nwin;
    return (int)(items < (long long)di.sms * per_sm ? items : (long long)di.sms * per_sm);
}

static int conv_tc5_fwd(const MmxConvHalfDesc* d, int data_gradient, const float* in, const float* w, const float* bias, float* out,
                        void* stream) {
    ctc5::ConvTc5Args a = conv_args(d);
    a.in = in; a.w = w; a.out = out; a.bias = data_gradient ? nullptr : bias;
    if (data_gradient) { a.transposed = 1; a.pt = d->kt - 1 - d->pad_t; a.pp = d->kp - 1 - d->pad_p; }
    const ctc5::ConvGeom g = ctc5::conv_tc5_geom(d->C, d->T, d->E, d->kt, d->kp);
    const size_t smem = ctc5::conv_tc5_smem(g, d->C, false).total;
    const int cols = 2 * g.NP <= 128 ? 128 : 2 * g.NP <= 256 ? 256 : 512;
    const int grid = conv_grid(g, d->B, smem, cols);
    if (cols == 128) return launch_tc5(ctc5::conv_tc5_fwd_kernel<128>, a, grid, tc5::kCtaThreads, smem, stream);
    if (cols == 256) return launch_tc5(ctc5::conv_tc5_fwd_kernel<256>, a, grid, tc5::kCtaThreads, smem, stream);
    return launch_tc5(ctc5::conv_tc5_fwd_kernel<512>, a, grid, tc5::kCtaThreads, smem, stream);
}

static int conv_tc5_wgrad(const MmxConvHalfDesc* d, const float* dz, const float* n, float* dw, float* db, void* stream) {
    ctc5::ConvTc5Args a = conv_args(d);
    a.in = n; a.dz = dz; a.dw = dw; a.db = db;
    const ctc5::ConvGeom g = ctc5::conv_tc5_geom(d->C, d->T, d->E, d->kt, d->kp);
    const size_t smem = ctc5::conv_tc5_smem(g, d->C, true).total;
    const int cols = (g.MR / 128) * g.Kp <= 128 ? 128 : 256;
    const int grid = conv_grid(g, d->B, smem, cols);
    if (cols == 128) return launch_tc5(ctc5::conv_tc5_wgrad_kernel<128>, a, grid, tc5::kCtaThreads, smem, stream);
    return launch_tc5(ctc5::conv_tc5_wgrad_kernel<256>, a, grid, tc5::kCtaThreads, smem, stream);
}
#endif

extern "C" int mmx_conv2d_tc5_serves(const MmxConvHalfDesc* d) { return conv_tc5_ok(d) ? 1 : 0; }

extern "C" int mmx_conv2d_large_fwd_prec(const MmxConvHalfDesc* d, int data_gradient, const float* in, const float* w, const float* bias,
                                         float* out, int precision, void* stream) {
    if (precision == MMX_PREC_TF32 && in && w && out && conv_tc5_ok(d)) return conv_tc5_fwd(d, data_gradient, in, w, bias, out, stream);
    return mmx_conv2d_large_fwd(d, data_gradient, in, w, bias, out, stream);
}

extern "C" int mmx_conv2d_large_wgrad_prec(const MmxConvHalfDesc* d, const float* dz, const float* n, float* dw, float* db, int precision,
                                           void* stream) {
    if (precision == MMX_PREC_TF32 && dz && n && dw && db && conv_tc5_ok(d)) return conv_tc5_wgrad(d, dz, n, dw, db, stream);
    return mmx_conv2d_large_wgrad(d, dz, n, dw, db, stream);
}
