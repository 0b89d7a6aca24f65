// mmx_mlp_block_fwd: fused MixerBlock forward (include/mmx.h).
#include "mmx_mlp_host.cuh"

using namespace mmx;

namespace mmx_tu_mlp_fwd {
template <int ACT, int TC, int TOKC>
struct MlpFwdBody { static MMX_D void run(Exec& ex, const MlpBlockFwdArgs& a) { mlp_block_fwd_body<ACT, TC, TOKC>(ex, a); } };

template <int ACT, int TC, int TOKC>
struct MlpFwdWarpBody { static MMX_D void run(Exec& ex, const MlpBlockFwdArgs& a) { mlp_block_fwd_warp_body<ACT, TC, TOKC>(ex, a); } };

template <int ACT>
int dispatch_mlp_fwd(const MlpBlockFwdArgs& a, int grid, size_t smem, void* stream) {
    if (a.d.T == 10 && a.d.tok == 20) return launch<MlpFwdBody<ACT, 10, 20>>(a, grid, kThreads, smem, stream);
    return launch<MlpFwdBody<ACT, 0, 0>>(a, grid, kThreads, smem, stream);
}
}  // namespace mmx_tu_mlp_fwd
using namespace mmx_tu_mlp_fwd;

bool mmx_mlp_tc5_ok(const MmxMlpBlockDesc* d);
int mmx_mlp_tc5_fwd(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const float* x, float* y, void* stream);

extern "C" int mmx_mlp_block_fwd(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const float* x, float* y, void* stream) {
    if (!x || !y) return fail(MMX_E_INVALID, "mmx_mlp_block_fwd: null tensor");
    MlpBlockFwdArgs a;
    size_t smem; int grid, nwarp = 0;
    if (!d) return fail(MMX_E_INVALID, "null descriptor");
    if (mmx_mlp_tc5_ok(d)) return mmx_mlp_tc5_fwd(d, w, x, y, stream);   // tcgen05 / TMEM family (sm_100a)
    const bool warp_variant = mlp_warp_variant_ok(d);
    int rc = warp_variant ? plan_mlp_block_warp(d, false, &a.d, &smem, &grid, &nwarp) : plan_mlp_block(d, false, &a.d, &smem, &grid);
    if (rc) return rc;
    if ((rc = check_block_params(w, d->use_se, "mmx_mlp_block_fwd"))) return rc;
    a.dr = make_dropout(d->dropout, d->training);
    a.w = to_w(w); a.x = x; a.y = y;
    if (warp_variant) {
        const int thr = nwarp * 32;
        // the 128-register build, two CTAs per SM (measured 8 % faster than 1 x 254 registers)
        return d->act == MMX_ACT_GELU ? launch<MlpFwdWarpBody<ACT_GELU, 10, 20>, MlpBlockFwdArgs, 2>(a, grid, thr, smem, stream)
                                      : launch<MlpFwdWarpBody<ACT_MISH, 10, 20>, MlpBlockFwdArgs, 2>(a, grid, thr, smem, stream);
    }
    return d->act == MMX_ACT_GELU ? dispatch_mlp_fwd<ACT_GELU>(a, grid, smem, stream) : dispatch_mlp_fwd<ACT_MISH>(a, grid, smem, stream);
}

int mmx_mlp_tc5_fwd_save(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const float* x, float* y, float* x1, float* gate, void* stream);
int mmx_mlp_tc5_bwd_saved(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const MmxMlpBlockParams* grads, const float* x,
                          const float* x1, const float* gate, const float* dy, float* dx, void* stream);

extern "C" int mmx_mlp_block_saves(const MmxMlpBlockDesc* d) { return d && mmx_mlp_tc5_ok(d) ? 1 : 0; }

extern "C" int mmx_mlp_block_fwd_save(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const float* x, float* y, float* x1, float* gate,
                                      void* stream) {
    if (!d) return fail(MMX_E_INVALID, "null descriptor");
    if (!x || !y) return fail(MMX_E_INVALID, "mmx_mlp_block_fwd_save: null tensor");
    if (!mmx_mlp_tc5_ok(d)) return fail(MMX_E_UNSUPPORTED, "mmx_mlp_block_fwd_save: shape / precision not served by the kernels that save the token-half output (see mmx_mlp_block_saves)");
    return mmx_mlp_tc5_fwd_save(d, w, x, y, x1, gate, stream);
}

extern "C" int mmx_mlp_block_bwd_saved(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const MmxMlpBlockParams* grads, const float* x,
                                       const float* x1, const float* gate, const float* dy, float* dx, void* stream) {
    if (!d) return fail(MMX_E_INVALID, "null descriptor");
    if (!x || !dy || !dx) return fail(MMX_E_INVALID, "mmx_mlp_block_bwd_saved: null tensor");
    if (!mmx_mlp_tc5_ok(d)) return fail(MMX_E_UNSUPPORTED, "mmx_mlp_block_bwd_saved: shape / precision not served (see mmx_mlp_block_saves)");
    return mmx_mlp_tc5_bwd_saved(d, w, grads, x, x1, gate, dy, dx, stream);
}
