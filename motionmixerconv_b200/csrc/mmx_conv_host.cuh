// Host-side planning (tile size, shared-memory budget, grid) for the ConvMixer kernels.
#pragma once
#include "mmx_launch.cuh"
#include "mmx_conv.cuh"

namespace mmx {

static inline ConvHalfW to_cw(const MmxConvHalfParams* p) {
    ConvHalfW w;
    w.ln_g = p->ln_w; w.ln_b = p->ln_b; w.cw = p->conv_w; w.cb = p->conv_b; w.se1 = p->se_w1; w.se2 = p->se_w2;
    return w;
}

static inline int check_conv_params(const MmxConvHalfParams* p, int use_se, const char* what) {
    if (!p) return fail(MMX_E_INVALID, "%s: null parameter table", what);
    if (!p->ln_w || !p->ln_b || !p->conv_w || !p->conv_b) return fail(MMX_E_INVALID, "%s: null parameter pointer", what);
    if (use_se && (!p->se_w1 || !p->se_w2)) return fail(MMX_E_INVALID, "%s: use_se set but SE weights are null", what);
    return MMX_OK;
}

// sequences per CTA tile: about kConvTileElems activations per tile, shrunk until the shared-memory layout fits
constexpr int kConvTileElems = 8192;

static inline int plan_conv_half(const MmxConvHalfDesc* d, bool bwd, ConvDims* out, size_t* smem, int* grid) {
    if (!d) return fail(MMX_E_INVALID, "null descriptor");
    if (d->B <= 0 || d->C <= 0 || d->T <= 0 || d->E <= 0 || d->kt <= 0 || d->kp <= 0) return fail(MMX_E_INVALID, "non-positive dimension");
    if (d->act != MMX_ACT_GELU && d->act != MMX_ACT_MISH) return fail(MMX_E_INVALID, "Unknown activation function type: %d", d->act);
    if (d->C > 8) return fail(MMX_E_UNSUPPORTED, "conv_nChan %d > 8", d->C);
    if (d->T > 32) return fail(MMX_E_UNSUPPORTED, "in_nTP %d > 32", d->T);
    if (d->pad_t < 0 || d->pad_p < 0 || d->pad_t > d->kt - 1 || d->pad_p > d->kp - 1)
        return fail(MMX_E_INVALID, "padding (%d,%d) does not keep the [T,E] shape for kernel (%d,%d)", d->pad_t, d->pad_p, d->kt, d->kp);
    if (d->use_se && d->se_hidden < 1) return fail(MMX_E_UNSUPPORTED, "in_nTP // r_se == 0: empty SE bottleneck");
    if (bwd && d->C * d->kt * ((d->kp + 3) / 4) > kThreads)
        return fail(MMX_E_UNSUPPORTED, "conv kernel %dx%dx(%d,%d) too large for the weight-gradient tiling", d->C, d->C, d->kt, d->kp);
    const DevInfo di = dev_info();
    ConvDims m;
    m.B = d->B; m.C = d->C; m.T = d->T; m.E = d->E; m.kT = d->kt; m.kP = d->kp; m.pT = d->pad_t; m.pP = d->pad_p;
    m.rr = d->use_se ? d->se_hidden : 0; m.use_se = d->use_se; m.use_max = d->use_max_pooling; m.training = d->training;
    m.site = d->site; m.bn_mode = 0;
    const int forced = env_int(bwd ? "MMX_CONV_S_BWD" : "MMX_CONV_S_FWD", 0);   // tests: force the tile
    // about kConvTileElems activations per tile, but never fewer tiles than ~2 per SM when the batch is small
    int S0 = imax(1, kConvTileElems / (d->C * d->T * d->E));
    S0 = imax(1, imin(S0, (d->B + 2 * di.sms - 1) / (2 * di.sms)));
    if (forced > 0) S0 = forced;
    for (int in_smem = 1; in_smem >= (bwd ? 0 : 1); --in_smem) {
        if (bwd && in_smem && env_int("MMX_CONV_X_GLOBAL", 0)) continue;   // tests: force the streamed-input variant
        m.x_in_smem = in_smem;
        const int S = fit_tile(di, S0, forced > 0 ? forced : 1, 1, true, [&](int s) { m.S = s; return (size_t)conv_smem(m, bwd).total * 4; });
        if (S) {
            m.S = imin(S, d->B);
            const size_t bytes = (size_t)conv_smem(m, bwd).total * 4;
            *out = m; *smem = bytes; *grid = tile_grid(di, d->B, m.S, bytes);
            return MMX_OK;
        }
    }
    return fail(MMX_E_UNSUPPORTED, "ConvMixerBlock tile does not fit shared memory (C=%d T=%d E=%d kernel %dx%d)", d->C, d->T, d->E, d->kt, d->kp);
}

}  // namespace mmx
