// Host-side planning (tile size, shared-memory budget, grid) for the MixerBlock kernels.
#pragma once
#include "mmx_launch.cuh"
#include "mmx_mlp.cuh"
#include "mmx_mlp_warp.cuh"

namespace mmx {
// ---------------------------------------------------------------------------------- MlpMixer block
static inline MlpBlockW to_w(const MmxMlpBlockParams* p) {
    MlpBlockW w;
    w.ln1_g = p->ln1_w; w.ln1_b = p->ln1_b; w.tw1 = p->tok_w1; w.tb1 = p->tok_b1; w.tw2 = p->tok_w2; w.tb2 = p->tok_b2;
    w.ln2_g = p->ln2_w; w.ln2_b = p->ln2_b; w.cw1 = p->ch_w1; w.cb1 = p->ch_b1; w.cw2 = p->ch_w2; w.cb2 = p->ch_b2;
    w.se1 = p->se_w1; w.se2 = p->se_w2;
    return w;
}

static inline int check_block_params(const MmxMlpBlockParams* p, int use_se, const char* what) {
    if (!p) return fail(MMX_E_INVALID, "%s: null parameter table", what);
    const float* v[] = {p->ln1_w, p->ln1_b, p->tok_w1, p->tok_b1, p->tok_w2, p->tok_b2, p->ln2_w, p->ln2_b, p->ch_w1, p->ch_b1, p->ch_w2, p->ch_b2};
    for (const float* q : v)
        if (!q) return fail(MMX_E_INVALID, "%s: null parameter pointer", what);
    if (use_se && (!p->se_w1 || !p->se_w2)) return fail(MMX_E_INVALID, "%s: use_se set but SE weights are null", what);
    return MMX_OK;
}

// choose sequences-per-tile and whether the channel-MLP weights live in shared memory
static inline int plan_mlp_block(const MmxMlpBlockDesc* d, bool bwd, MlpDims* out, size_t* smem, int* grid) {
    if (!d) return fail(MMX_E_INVALID, "null descriptor");
    if (d->B <= 0 || d->T <= 0 || d->H <= 0 || d->tok <= 0 || d->ch <= 0) return fail(MMX_E_INVALID, "non-positive dimension");
    if (d->act != MMX_ACT_GELU && d->act != MMX_ACT_MISH) return fail(MMX_E_INVALID, "Unknown activation function type: %d", d->act);
    if (d->T > 32 || d->tok > 64) return fail(MMX_E_UNSUPPORTED, "seq_len %d > 32 or tokens_mlp_dim %d > 64", d->T, d->tok);
    if (d->use_se && d->se_hidden < 1) return fail(MMX_E_UNSUPPORTED, "seq_len // r_se == 0: empty SE bottleneck");
    const DevInfo di = dev_info();
    MlpDims m;
    m.B = d->B; m.T = d->T; m.H = d->H; m.tok = d->tok; m.ch = d->ch; m.rr = d->use_se ? d->se_hidden : 0;
    m.use_se = d->use_se; m.use_max = d->use_max_pooling; m.training = d->training; m.site_base = d->block_index * 4;
    const int row_target = bwd ? 96 : 128;
    // Two candidates: channel-MLP weights staged in shared memory, or read from global (L1/L2; needs H, ch % 4 == 0).  Large H:
    // the staged weights leave room for a single sequence per tile (10 rows: GEMM phases with a handful of busy threads),
    // so take the global-weights layout when it at least doubles the rows per tile.
    int bestS[2] = {0, 0};
    for (int in_smem = 1; in_smem >= 0; --in_smem) {
        if (!in_smem && ((d->H & 3) || (d->ch & 3))) continue;
        m.w_in_smem = in_smem;
        bestS[in_smem] = fit_tile(di, imax(1, row_target / d->T), 1, 1, true, [&](int S) { m.S = S; return (size_t)mlp_block_smem(m, bwd).total * 4; });
    }
    int pick = bestS[1] ? 1 : 0;
    if (bestS[0] >= 2 * imax(bestS[1], 1) && bestS[1] * d->T < 32) pick = 0;
    if (bestS[pick]) {
        m.w_in_smem = pick;
        m.S = imin(bestS[pick], d->B);
        if (m.S == bestS[pick] && m.S >= 2) m.S = balanced_tile(d->B, m.S, (m.S + 1) / 2, 1, di.sms);
        const size_t bytes = (size_t)mlp_block_smem(m, bwd).total * 4;
        *out = m; *smem = bytes; *grid = tile_grid(di, d->B, m.S, bytes);
        return MMX_OK;
    }
    return fail(MMX_E_UNSUPPORTED, "MixerBlock tile does not fit shared memory (H=%d ch=%d)", d->H, d->ch);
}

// ---------------------------------------------------------------------------------- warp-per-sequence-pair variant
constexpr int kWarpVariantWarps = 8;

static inline bool mlp_warp_variant_ok(const MmxMlpBlockDesc* d) {
    return d->T == 10 && d->tok == 20 && d->H <= 64 && d->ch <= 64 && !d->use_max_pooling && !env_int("MMX_MLP_V1", 0);
}

static inline int plan_mlp_block_warp(const MmxMlpBlockDesc* d, bool bwd, MlpDims* out, size_t* smem, int* grid, int* nwarp_out) {
    if (d->B <= 0) return fail(MMX_E_INVALID, "non-positive dimension");
    if (d->act != MMX_ACT_GELU && d->act != MMX_ACT_MISH) return fail(MMX_E_INVALID, "Unknown activation function type: %d", d->act);
    if (d->use_se && d->se_hidden < 1) return fail(MMX_E_UNSUPPORTED, "seq_len // r_se == 0: empty SE bottleneck");
    const DevInfo di = dev_info();
    MlpDims m;
    m.B = d->B; m.T = d->T; m.H = d->H; m.tok = d->tok; m.ch = d->ch; m.rr = d->use_se ? d->se_hidden : 0;
    m.use_se = d->use_se; m.use_max = 0; m.training = d->training; m.site_base = d->block_index * 4;
    m.S = kSPW; m.w_in_smem = 1;
    int nwarp = kWarpVariantWarps;
    size_t bytes = 0;
    for (; nwarp >= 2; --nwarp) {      // as many warps per CTA as the shared-memory scratch allows
        bytes = (size_t)mlp_warp_smem(m, bwd, nwarp).total * 4;
        if (bytes <= (size_t)di.max_smem) break;
    }
    if (nwarp < 2) return fail(MMX_E_UNSUPPORTED, "MixerBlock (warp variant) does not fit shared memory");
    const int per_sm = ctas_per_sm(di, bytes, 4);
    const int groups = (d->B + kSPW - 1) / kSPW;
    const int max_warps = di.sms * per_sm * nwarp;
    const int waves = (groups + max_warps - 1) / max_warps;
    const int warps_needed = (groups + waves - 1) / waves;
    // spread the warps over every CTA slot of the device (fewer warps per CTA) instead of filling fewer CTAs: a warp runs
    // faster with fewer co-resident warps and the makespan is waves x the per-pair latency either way
    const int slots = di.sms * per_sm;
    const int spread = imax(2, imin(nwarp, (warps_needed + slots - 1) / slots));
    if (spread < nwarp) {
        nwarp = spread;
        bytes = (size_t)mlp_warp_smem(m, bwd, nwarp).total * 4;
    }
    *out = m; *smem = bytes; *grid = imax(1, (warps_needed + nwarp - 1) / nwarp); *nwarp_out = nwarp;
    return MMX_OK;
}

}  // namespace mmx
