/* libmmx — C ABI of the B200 (sm_100a) ConvMixer / MotionMixer hot path.
 *
 * The reference (AlekseiZhuravlev/MotionMixerConv) is pure Python/PyTorch and has no FFI of its
 * own: its "plugin interface" for this path is the nn.Module surface
 *     h36m/mlp_mixer.py:254-258,306        MlpMixer(...).forward(x)
 *     h36m/conv_mixer_model.py:357-379,428 ConvMixer(...).forward(x)
 *     h36m/utils/utils_mixer.py:48         mpjpe_error(pred, gt)
 *     h36m/train_mixer_h36m.py:63,193      optim.Adam(...).step()
 * The Python package motionmixerconv_b200 mirrors that surface and binds the entry points below
 * with ctypes (INTEGRATION.md shows the stub).  Each entry point cites the reference code whose
 * arithmetic it replaces.
 *
 * Conventions: all tensors fp32, contiguous, row-major, DEVICE pointers borrowed from the caller
 * (torch's caching allocator).  Nothing here allocates, frees or synchronises; kernels are
 * enqueued on `stream` (a cudaStream_t) of the CURRENT device.  Gradient outputs are
 * ACCUMULATED (+=, RED.ADD) so the caller zeroes them once per step.  Return value: 0 on
 * success, negative on error (MMX_E_*); mmx_last_error() gives a thread-local message.
 */
#ifndef MMX_H_
#define MMX_H_

#ifdef __cplusplus
extern "C" {
#endif

#define MMX_OK 0
#define MMX_E_INVALID (-1)     /* bad argument (null pointer, non-positive size, ...) */
#define MMX_E_UNSUPPORTED (-2) /* shape outside what the kernels are built for */
#define MMX_E_CUDA (-3)        /* CUDA runtime error (message has the cudaError string) */

#define MMX_ACT_GELU 0
#define MMX_ACT_MISH 1

/* Arithmetic of the contractions inside a fused block.  FP32: fp32 FMA everywhere (1e-5 parity with the reference).
 * TF32 (the reduced-precision "bf16/TF32" mode, 2e-3 parity): the channel-MLP contractions run on the tensor cores --
 * tcgen05.mma on bf16 operands split hi + lo (three MMAs per product, fp32 accumulation in TMEM) where the tcgen05 family
 * serves the shape, mma.sync TF32 otherwise; LayerNorm, activations, SE, residuals and every reduction stay fp32.
 * It is a permission: shapes no tensor-core kernel serves run FP32. */
#define MMX_PREC_FP32 0
#define MMX_PREC_TF32 1

int mmx_version(void);
const char* mmx_last_error(void);

/* Dropout (nn.Dropout sites inside the blocks; mlp_mixer.py:68-70, conv_mixer_model.py:113-114).  p == 0 disables.  Masks are a
 * pure function of (seed, site, step + *step_dev, element); the generator depends on the kernel family serving the shape
 * (tests/masks_np.py holds bit-exact numpy twins of all of them):
 *   generic MixerBlock / ConvMixer kernels: Philox4x32-10, one 32-bit word per element;
 *   warp-per-sequence-pair MixerBlock kernels: Philox4x32-7, 16 bits per element;
 *   tcgen05 MixerBlock kernels: lowbias32 counter hash, 16 bits per element. */
typedef struct {
    float p;
    unsigned long long seed;
    unsigned int step;            /* host-side step counter ...                                   */
    const unsigned int* step_dev; /* ... plus (if non-null) a DEVICE counter read by the kernel, so a
                                     launch recorded in a CUDA graph draws fresh masks on every replay */
} MmxDropout;

/* ---------------- MlpMixer (h36m/mlp_mixer.py) ---------------- */

/* One MixerBlock (mlp_mixer.py:100-164).  Parameter pointers use the reference layouts. */
typedef struct {
    float *ln1_w, *ln1_b;   /* LN1.weight, LN1.bias                               [H]          */
    float *tok_w1, *tok_b1; /* mlp_block_token_mixing.fc1.{weight,bias}           [tok,T],[tok]*/
    float *tok_w2, *tok_b2; /* mlp_block_token_mixing.fc2.{weight,bias}           [T,tok],[T]  */
    float *ln2_w, *ln2_b;   /* LN2.weight, LN2.bias                               [H]          */
    float *ch_w1, *ch_b1;   /* mlp_block_channel_mixing.fc1.{weight,bias}         [ch,H],[ch]  */
    float *ch_w2, *ch_b2;   /* mlp_block_channel_mixing.fc2.{weight,bias}         [H,ch],[H]   */
    float *se_w1, *se_w2;   /* se.excitation.0.weight [T/r,T], se.excitation.2.weight [T,T/r]; null if !use_se */
} MmxMlpBlockParams;

typedef struct {
    int B, T, H, tok, ch; /* batch, seq_len, hidden_dim, tokens_mlp_dim, channels_mlp_dim */
    int se_hidden;        /* T / r_se */
    int act;              /* MMX_ACT_* */
    int use_se, use_max_pooling;
    int training;         /* dropout active only when training != 0 */
    int block_index;      /* selects the dropout sites of this block */
    MmxDropout dropout;
    int precision;        /* MMX_PREC_* */
} MmxMlpBlockDesc;

/* y = MixerBlock(x): LN1 -> token MLP -> SE -> +res -> LN2 -> channel MLP -> SE -> +res, fused.
 * Replaces MixerBlock.forward, mlp_mixer.py:138-164. x,y: [B,T,H]. */
int mmx_mlp_block_fwd(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const float* x, float* y, void* stream);
/* Backward of the same (autograd of mlp_mixer.py:138-164); the forward is recomputed from x.
 * dx: [B,T,H] written; grads: accumulated. */
int mmx_mlp_block_bwd(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const MmxMlpBlockParams* grads,
                      const float* x, const float* dy, float* dx, void* stream);

/* Variant that trades one saved tile for less backward work (used by the autograd Function and TrainStep when available):
 * the forward also writes x1 = x + SE(token MLP(LN1 x)) [B,T,H] (the input of the block's channel half, mlp_mixer.py:155) and
 * its SE gates [B,T] (null without SE); the backward then skips the token-half forward and the token-MLP recompute.
 * mmx_mlp_block_saves: 1 when the kernels serving this descriptor support it (the tcgen05 family), else 0. */
int mmx_mlp_block_saves(const MmxMlpBlockDesc* d);
int mmx_mlp_block_fwd_save(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const float* x, float* y, float* x1, float* gate, void* stream);
int mmx_mlp_block_bwd_saved(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const MmxMlpBlockParams* grads,
                            const float* x, const float* x1, const float* gate, const float* dy, float* dx, void* stream);

/* The two halves of a MixerBlock as the tcgen05 family runs them (MMX_E_UNSUPPORTED when mmx_mlp_block_saves(d) == 0):
 *   token half   (mlp_mixer.py:146-155)  x1 = x + SE(token MLP(LN1 x)^T)^T          fp32 CUDA cores (packed fma.rn.f32x2)
 *   channel half (mlp_mixer.py:157-164)  y  = x1 + SE(channel MLP(LN2 x1))          tcgen05.mma, accumulators in TMEM
 * token_half_bwd: x1 / gate nullable (then the token MLP output is recomputed); dx may alias dx1.  channel_half_bwd: dx1 may
 * alias x1.  Gradients accumulated. */
int mmx_mlp_token_half_fwd(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const float* x, float* x1, float* gate, void* stream);
int mmx_mlp_token_half_bwd(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const MmxMlpBlockParams* grads, const float* x,
                           const float* x1, const float* gate, const float* dx1, float* dx, void* stream);
int mmx_mlp_channel_half_fwd(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const float* x1, float* y, void* stream);
int mmx_mlp_channel_half_bwd(const MmxMlpBlockDesc* d, const MmxMlpBlockParams* w, const MmxMlpBlockParams* grads, const float* x1,
                             const float* dy, float* dx1, void* stream);

/* ---- MixerBlock with regularization == -1: BatchNorm1d inside the MLP blocks (mlp_mixer.py:72-73 reg1 / reg2, applied at :90-94) ----
 * Batch statistics are global over the batch, so the block runs as a chain of stage kernels sequenced by the caller
 * (motionmixerconv_b200/functional.py MlpBnBlock); the fc layers are mmx_linear_{fwd,bwd}:
 *   token half  : ln_fwd (Tt = T: output transposed [B,H,T]) -> fc1 -> bn1d_stats/finalize/apply (act) -> fc2 -> bn1d_stats/finalize
 *                 -> se_res_fwd (v transposed, affine per h)                              BatchNorm1d(hidden_dim): [N,C,L] = [B,H,*]
 *   channel half: ln_fwd -> fc1 -> bn1d_stats/finalize/apply (act) -> fc2 -> bn1d_stats/finalize -> se_res_fwd (affine per t)
 *                                                                                          BatchNorm1d(seq_len):    [N,C,L] = [B,T,*]
 * and the backward mirrors it: se_res_bwd -> bn1d_bwd_reduce / mmx_bn_coef / bn1d_bwd_apply -> fc2 bwd -> ... -> ln_bwd.
 * Per-channel vectors as in the ConvMixer BatchNorm path: bn = [scale|shift|xs|xo][C] (mmx_bn_finalize), coef = [k1|k2|k3][C]
 * (mmx_bn_coef).  act: MMX_ACT_* (the statistic is taken AFTER the activation, u is the pre-activation) or -1 (identity). */
/* y = LayerNorm(x) over rows of width H (eps 1e-5); stats[r] = (mean, rstd).  Tt > 0: row r = (b, t) of [B,Tt,H] and y is
 * written transposed, y[b][h][t]  (mlp_mixer.py:146-149). */
int mmx_ln_fwd(long long rows, int H, int Tt, const float* x, const float* g, const float* b, float* y, float* stats, void* stream);
/* dx = res (nullable) + LayerNorm backward of dy (Tt > 0: dy laid out [B][H][Tt]); dg, db accumulated.  dx may alias res. */
int mmx_ln_bwd(long long rows, int H, int Tt, const float* x, const float* stats, const float* g, const float* dy, const float* res,
               float* dx, float* dg, float* db, void* stream);
/* u: [N,C,L].  sums[0:C] += sum_{n,l} a, sums[C:2C] += sum a^2, a = act(u)  (then mmx_bn_finalize with n = N*L). */
int mmx_bn1d_stats(long long N, int C, int L, int act, const float* u, double* sums, void* stream);
/* y = act(u) * scale[c] + shift[c]  (bn[0:C], bn[C:2C]; eval mode: the running-statistics affine). */
int mmx_bn1d_apply(long long N, int C, int L, int act, const float* u, const float* bn, float* y, void* stream);
/* sums[0:C] += sum dy, sums[C:2C] += sum dy * xhat, xhat = act(u)*xs[c] + xo[c]  (then mmx_bn_coef). */
int mmx_bn1d_bwd_reduce(long long N, int C, int L, int act, const float* u, const float* bn, const float* dy, double* sums, void* stream);
/* du = k1[c] * (dy - k2[c] - xhat*k3[c]) * act'(u); du may alias dy. */
int mmx_bn1d_bwd_apply(long long N, int C, int L, int act, const float* u, const float* bn, const float* coef, const float* dy,
                       float* du, void* stream);
/* out = x + SE(y), y = v*scale + shift (the second BatchNorm of the MlpBlock folded in; mlp_mixer.py:152-155, 161-164, SELayer
 * :30-34).  x, out: [B,T,H]; v: [B,T,H] or, v_transposed, [B,H,T]; the affine is indexed by h (affine_by_h, token half) or by t.
 * se_hidden == 0: no SE (gate 1). */
int mmx_se_res_fwd(int B, int T, int H, int se_hidden, int use_max_pooling, int v_transposed, int affine_by_h, const float* x,
                   const float* v, const float* bn, const float* se_w1, const float* se_w2, float* out, void* stream);
/* dv (v's layout) = gradient wrt y of the same; SE weight gradients accumulated.  (The residual's gradient is dout itself.) */
int mmx_se_res_bwd(int B, int T, int H, int se_hidden, int use_max_pooling, int v_transposed, int affine_by_h, const float* v,
                   const float* bn, const float* se_w1, const float* se_w2, const float* dout, float* g_se_w1, float* g_se_w2,
                   float* dv, void* stream);

/* Diagnostics of the tcgen05 / TMEM MixerBlock kernels (precision == MMX_PREC_TF32): number of kernels whose mbarrier waits
 * timed out since the process started (a mis-programmed pipeline ends the kernel instead of hanging the GPU); 0 in a healthy
 * run.  Synchronises the device. */
int mmx_tc5_abort_count(void);
/* Test / debug: the keep-scales (0 or 1/(1-p)) the tcgen05 MixerBlock kernels draw for dropout site `site` seen as a
 * [rows][W] tensor (d->step_dev is ignored).  Channel MLP: site 4*block+2 on [B*T][ch], 4*block+3 on [B*T][H]; token MLP: ONE
 * stream per (sequence, hidden column), site 4*block on [B*H][tok+T] (columns [0,tok): after the activation, the rest: after fc2).
 * tests/masks_np.py holds the numpy twin. */
int mmx_tc5_dropout_mask(const MmxDropout* d, unsigned int site, long long rows, int W, float* out, void* stream);

/* y[r,:] = W x[r,:] + b  — MlpMixer.conv (Conv2d(1,H,(1,D)) == per-frame Linear, mlp_mixer.py:268,325-327)
 * and PoseEncoder.embed_mlp without harmonics (positional_encoder.py:91).  x:[rows,K] w:[N,K] y:[rows,N]. */
int mmx_linear_fwd(int rows, int K, int N, const float* x, const float* w, const float* b, float* y, void* stream);
/* dw,db accumulated; dx (may be null) written. */
int mmx_linear_bwd(int rows, int K, int N, const float* x, const float* w, const float* dy, float* dw, float* db,
                   float* dx, void* stream);
/* The same with a precision mode (MMX_PREC_*): MMX_PREC_TF32 runs the layer on the tensor cores (tcgen05, bf16 hi+lo split
 * operands, fp32 accumulation; measured error ~1e-5 relative) when the shape is served (K+1, N <= 80, even; 16-byte aligned
 * tensors), and falls back to the fp32 kernels otherwise.  The plain entry points above are precision MMX_PREC_FP32. */
int mmx_linear_fwd_prec(int rows, int K, int N, const float* x, const float* w, const float* b, float* y, int precision, void* stream);
int mmx_linear_bwd_prec(int rows, int K, int N, const float* x, const float* w, const float* dy, float* dw, float* db,
                        float* dx, int precision, void* stream);

typedef struct {
    float *ln_w, *ln_b;  /* LN.weight, LN.bias            [H]            */
    float *wt, *bt;      /* conv_out.weight [To,T,1], conv_out.bias [To] */
    float *wf, *bf;      /* fc_out.weight [D,H], fc_out.bias [D]         */
} MmxMlpHeadParams;
typedef struct { int B, T, To, H, D; } MmxMlpHeadDesc;

/* out = fc_out(conv_out(LN(x)))  — mlp_mixer.py:332-335.  x:[B,T,H] out:[B,To,D]. */
int mmx_mlp_head_fwd(const MmxMlpHeadDesc* d, const MmxMlpHeadParams* w, const float* x, float* out, void* stream);
int mmx_mlp_head_bwd(const MmxMlpHeadDesc* d, const MmxMlpHeadParams* w, const MmxMlpHeadParams* grads,
                     const float* x, const float* dout, float* dx, void* stream);
/* The same with a precision mode: MMX_PREC_TF32 runs the whole head as one tcgen05 kernel per direction (H < 64, D <= 80,
 * H and D even and >= 8, T, To <= 128, T*H and To*D multiples of 4, 16-byte aligned tensors), see csrc/mmx_head_tc5.cuh;
 * other shapes fall back to the fp32 kernels, which serve T <= 32 (MMX_E_UNSUPPORTED above). */
int mmx_mlp_head_fwd_prec(const MmxMlpHeadDesc* d, const MmxMlpHeadParams* w, const float* x, float* out, int precision, void* stream);
int mmx_mlp_head_bwd_prec(const MmxMlpHeadDesc* d, const MmxMlpHeadParams* w, const MmxMlpHeadParams* grads,
                          const float* x, const float* dout, float* dx, int precision, void* stream);

/* ---------------- ConvMixer (h36m/conv_mixer_model.py, conv_mixer/encoding/positional_encoder.py) ---------------- */

/* One half of a ConvMixerBlock (conv_mixer_model.py:279-284 resp. :287-292):
 *     y = x + SE(reg(act(conv2d(LN(x)))))        x, y: [B, C, T, E]
 * conv: C -> C channels, kernel (kt, kp) over (time, embedding), stride 1, zero padding pad_t rows on top
 * and pad_p columns on the left (bottom / right = k-1-pad: PyTorch 'same' puts the surplus there; an explicit
 * padding tuple must satisfy 2*pad == k-1, otherwise the reference's residual add fails as well). */
typedef struct {
    float *ln_w, *ln_b;     /* LN1 / LN2 .weight, .bias                         [E]            */
    float *conv_w, *conv_b; /* conv1 / conv2 .conv.weight, .conv.bias           [C,C,kt,kp],[C]*/
    float *se_w1, *se_w2;   /* se.excitationBlock.0.weight [T/r,T], .2.weight [T,T/r]; null if !use_se */
    float* bn_aff;          /* eval-mode BatchNorm2d (conv{1,2}.reg) folded to a per-channel affine applied after the
                               activation: [scale[C] | shift[C]], scale = weight/sqrt(running_var+eps),
                               shift = bias - running_mean*scale; null: no BatchNorm.  Ignored in grads tables. */
} MmxConvHalfParams;

typedef struct {
    int B, C, T, E;         /* batch, conv_nChan, in_nTP, dimPosEmb */
    int kt, kp, pad_t, pad_p;
    int se_hidden;          /* T / r_se */
    int act;                /* MMX_ACT_* */
    int use_se, use_max_pooling;
    int training;
    int site;               /* dropout site of this half: 2*block_index + (0|1) */
    MmxDropout dropout;
} MmxConvHalfDesc;

int mmx_conv_half_fwd(const MmxConvHalfDesc* d, const MmxConvHalfParams* w, const float* x, float* y, void* stream);
/* dx written; grads accumulated.  The forward is recomputed from x. */
int mmx_conv_half_bwd(const MmxConvHalfDesc* d, const MmxConvHalfParams* w, const MmxConvHalfParams* grads,
                      const float* x, const float* dy, float* dx, void* stream);

/* Capability query: MMX_OK (+ sequences per CTA tile and dynamic shared memory of the plan) when mmx_conv_half_{fwd,bwd} serve
 * this descriptor, otherwise the error code they would return (mmx_last_error() says why).  No launch.
 * tools/conv_support_table.py tabulates the reference's Optuna grid (optuna_search/conv_optuna_main.py:339-342) with it. */
int mmx_conv_half_plan(const MmxConvHalfDesc* d, int backward, int* seq_per_tile, int* smem_bytes);

/* ---- large ConvMixerBlock halves: shapes whose tile does not fit the fused kernels (mmx_conv_half_plan says so: C = 8, E = 192 with
 * 5x9 ... 9x29 kernels, most of optuna_search/conv_optuna_main.py:339-342), and BatchNorm with the max squeeze.  Same arithmetic as
 * mmx_conv_half_{fwd,bwd}, as a chain of stage kernels with the intermediates in HBM (functional.ConvHalfLarge sequences them):
 *   forward :  mmx_ln_fwd -> mmx_conv2d_large_fwd -> [mmx_bn1d_stats (act) + mmx_bn_finalize] -> mmx_conv_tail_fwd
 *   backward:  mmx_conv_tail_bwd1 -> [mmx_bn_coef] -> mmx_conv_tail_bwd2 -> mmx_conv2d_large_fwd(data_gradient) + mmx_conv2d_large_wgrad
 *              -> mmx_ln_bwd
 * The descriptor is the half's MmxConvHalfDesc.  Dropout masks are those of the fused kernels. */
/* out = conv2d(in) + bias (conv_mixer_model.py:133); data_gradient != 0: d(in) from d(out) (weights flipped / transposed, no bias) */
int mmx_conv2d_large_fwd(const MmxConvHalfDesc* d, int data_gradient, const float* in, const float* w, const float* bias, float* out,
                         void* stream);
/* dw [C,C,kt,kp] += dz (*) n, db [C] += sum dz */
int mmx_conv2d_large_wgrad(const MmxConvHalfDesc* d, const float* dz, const float* n, float* dw, float* db, void* stream);
/* The same two convolutions with a precision mode.  MMX_PREC_TF32 runs them on the tensor cores (tcgen05, bf16 hi+lo split
 * operands, three MMAs per product, fp32 accumulation in TMEM; csrc/mmx_conv_tc5.cuh) when mmx_conv2d_tc5_serves(d); MMX_PREC_FP32
 * and every shape it does not serve give exactly the entry points above.  Served: 1 <= C <= 8, C * round_up(kp, 8) <= 256,
 * kt * C <= 128, kp <= 121 and the tile (the padded input slab of one sequence and 128 embedding positions, (T-1)*C +
 * round_up(kt*C, 16) rows) within shared memory -- at T = 10, E any, every kernel of the Optuna grid up to 9x29 at C = 8.
 * Plain loads and stores: no alignment beyond that of float. */
int mmx_conv2d_large_fwd_prec(const MmxConvHalfDesc* d, int data_gradient, const float* in, const float* w, const float* bias,
                              float* out, int precision, void* stream);
int mmx_conv2d_large_wgrad_prec(const MmxConvHalfDesc* d, const float* dz, const float* n, float* dw, float* db,
                                int precision, void* stream);
/* 1 when precision MMX_PREC_TF32 runs this descriptor's convolutions (fwd, data gradient, wgrad) on tcgen05; 0 otherwise.  No launch. */
int mmx_conv2d_tc5_serves(const MmxConvHalfDesc* d);
/* y = x + SE(reg(act(z))); reg = dropout of the descriptor, or (bn_aff != null) the BatchNorm affine [scale|shift][C] */
int mmx_conv_tail_fwd(const MmxConvHalfDesc* d, const float* x, const float* z, const float* bn_aff, const float* se_w1, const float* se_w2,
                      float* y, void* stream);
/* SE backward: gd [B,T,3] = (gate, d squeeze, argmax), SE weight gradients accumulated; bn ([scale|shift|xs|xo][C]) != null:
 * sums[0:C] += sum dR, sums[C:2C] += sum dR*xhat */
int mmx_conv_tail_bwd1(const MmxConvHalfDesc* d, const float* z, const float* dy, const float* bn, const float* se_w1, const float* se_w2,
                       float* g_se_w1, float* g_se_w2, float* gd, double* sums, void* stream);
/* dz [B,C,T,E] (gradient wrt the conv output) from dy, gd and, BatchNorm, bn + coef */
int mmx_conv_tail_bwd2(const MmxConvHalfDesc* d, const float* z, const float* dy, const float* gd, const float* bn, const float* coef,
                       float* dz, void* stream);

/* Training-mode BatchNorm2d between the activation and the SE layer (regularization == -1, conv_mixer_model.py:115-116,
 * 139-141) needs batch-global statistics, so a half runs as two passes each way; the per-channel vectors between the
 * passes are computed by the caller from the sums (a handful of C-element tensor ops):
 *   forward : bn_stats (LN -> conv; writes the pre-activation z [B,C,T,E]; sums[0:C] += sum act(z), sums[C:2C] += sum act(z)^2)
 *             bn_apply (y = x + SE(act(z)*scale + shift))
 *   backward: bn_bwd1  (SE backward; gd[b][t] = (gate, d pool); sums[0:C] += sum dR, sums[C:2C] += sum dR*xhat)
 *             bn_bwd2  (dA = k1*(dR - k2 - xhat*k3); conv / LN backward without recomputing the conv; dx written)
 * bn   = [scale | shift | xs | xo][C]:  R = act(z)*scale + shift,  xhat = act(z)*xs + xo  (xs = rstd, xo = -mean*rstd)
 * coef = [k1 | k2 | k3][C]:            k1 = weight*rstd, k2 = mean(dR), k3 = mean(dR*xhat)
 * SE gradients are accumulated by bn_bwd1, LN / conv gradients by bn_bwd2.  Mean squeeze only. */
int mmx_conv_half_bn_stats(const MmxConvHalfDesc* d, const MmxConvHalfParams* w, const float* x, float* z, double* sums, void* stream);
int mmx_conv_half_bn_apply(const MmxConvHalfDesc* d, const MmxConvHalfParams* w, const float* bn, const float* x, const float* z,
                           float* y, void* stream);
int mmx_conv_half_bn_bwd1(const MmxConvHalfDesc* d, const MmxConvHalfParams* w, const MmxConvHalfParams* grads, const float* bn,
                          const float* z, const float* dy, float* gd, double* sums, void* stream);
int mmx_conv_half_bn_bwd2(const MmxConvHalfDesc* d, const MmxConvHalfParams* w, const MmxConvHalfParams* grads, const float* bn,
                          const float* coef, const float* x, const float* z, const float* dy, const float* gd, float* dx,
                          void* stream);

/* BatchNorm bookkeeping between the passes (nn.BatchNorm2d semantics; C elements, one tiny launch each instead of ~25 tensor ops):
 * bn_finalize: sums -> bn = [scale|shift|xs|xo]; running_mean/var updated (momentum, unbiased variance), num_batches_tracked += 1;
 * bn_coef:     backward sums -> coef = [k1|k2|k3]; g_weight += sum dR*xhat, g_bias += sum dR.  Both zero `sums` on exit (the
 * accumulating kernels must start from zero).  n = elements per channel (B*T*E).  Any C (one thread per channel). */
int mmx_bn_finalize(double* sums, int C, double n, const float* w, const float* b, float* running_mean, float* running_var,
                    long long* num_batches_tracked, float momentum, float eps, float* bn, void* stream);
int mmx_bn_coef(double* sums, int C, double n, const float* bn, float* coef, float* g_weight, float* g_bias, void* stream);

/* mode_conv="once": the second half of ConvMixerBlock.forward degenerates to y = x + se(x)  (or 2x without SE),
 * conv_mixer_model.py:259-263,287-292.  x, y: [B,C,T,E]; se weights may be null when !use_se. */
int mmx_se_tail_fwd(int B, int C, int T, int E, int se_hidden, int use_se, int use_max_pooling,
                    const float* se_w1, const float* se_w2, const float* x, float* y, void* stream);
int mmx_se_tail_bwd(int B, int C, int T, int E, int se_hidden, int use_se, int use_max_pooling,
                    const float* se_w1, const float* se_w2, float* g_se_w1, float* g_se_w2,
                    const float* x, const float* dy, float* dx, void* stream);

/* PoseEncoder.forward (positional_encoder.py:79-97): optional harmonic embedding (sin/cos of x*frequencies,
 * the argument formed by ONE fp32 multiply) -> embed_mlp -> channelUpscaling.
 * x: [B,T,D];  m: [B*T,E] = embed_mlp output (saved for the backward);  y: [B,C,T,E]. */
typedef struct {
    float* freq;            /* encoder.frequencies [n_harmonic] (null when n_harmonic <= 0)                 */
    float *w, *b;           /* encoder.embed_mlp.weight [E, K], .bias [E];  K = n_harmonic>0 ? 2*n_harmonic*D : D */
    float *wc, *bc;         /* encoder.channelUpscaling.weight [C,1], .bias [C]                              */
} MmxEncoderParams;
typedef struct { int B, T, D, E, C, n_harmonic; } MmxEncoderDesc;

int mmx_pose_encoder_fwd(const MmxEncoderDesc* d, const MmxEncoderParams* w, const float* x, float* m, float* y, void* stream);
/* grads accumulated (grads->freq ignored).  dm_ws: caller-provided workspace [B*T,E].  dx: nullable; written. */
int mmx_pose_encoder_bwd(const MmxEncoderDesc* d, const MmxEncoderParams* w, const MmxEncoderParams* grads,
                         const float* x, const float* m, const float* dy, float* dm_ws, float* dx, void* stream);

/* ConvMixer head (conv_mixer_model.py:455-463): LN -> conv_out (T -> To) -> project_channels (C -> 1) -> GELU -> fc_out.
 * y: [B,C,T,E] -> out: [B,To,D]. */
typedef struct {
    float *ln_w, *ln_b;     /* LN.weight, LN.bias                              [E]             */
    float *wt, *bt;         /* conv_out.weight [To,T,1,1], conv_out.bias [To]                  */
    float *wp, *bp;         /* project_channels.weight [1,C,1,1], .bias [1]                    */
    float *wf, *bf;         /* fc_out.weight [D,E], fc_out.bias [D]                            */
} MmxConvHeadParams;
typedef struct { int B, C, T, To, E, D; } MmxConvHeadDesc;

int mmx_conv_head_fwd(const MmxConvHeadDesc* d, const MmxConvHeadParams* w, const float* y, float* out, void* stream);
int mmx_conv_head_bwd(const MmxConvHeadDesc* d, const MmxConvHeadParams* w, const MmxConvHeadParams* grads,
                      const float* y, const float* dout, float* dy, void* stream);

/* ---------------- the callers either side of model(x) ---------------- */

/* Step input (train_mixer_h36m.py:117-120,179): x = batch[:, :T, dim_used] * x_scale, gt = batch[:, T:T+To, dim_used] * gt_scale.
 * batch: [B,Ttot,Dfull], dim_used: DEVICE int32 [D], x: [B,T,D], gt: [B,To,D]. */
int mmx_window_split(const float* batch, int B, int Ttot, int Dfull, const int* dim_used, int D, int T, int To,
                     float x_scale, float gt_scale, float* x, float* gt, void* stream);

/* PCK histogram for auc_pck_metric (utils/utils_mixer.py:20-45): hist[k] += #joints with thresh[k-1] < ||pred-gt|| <= thresh[k]
 * (k = 0: <= thresh[0]; k = n: > thresh[n-1]); PCK(thresh[k]) = cumsum(hist)[k] / n_joints.  hist: DEVICE int32 [n+1], accumulated. */
int mmx_pck_hist(const float* pred, const float* gt, long long n_joints, const float* thresh, int n, int* hist, void* stream);

/* ---------------- loss / optimiser ---------------- */

/* MPJPE (utils_mixer.py:48-53): *loss_sum += sum_joints ||gt - pred||_2 (caller zeroes it; mean =
 * loss_sum / n_joints); dpred (nullable) = gscale * dL/dpred of the MEAN, 0 at zero distance. */
int mmx_mpjpe_fwd_bwd(const float* pred, const float* gt, float* dpred, float* loss_sum, long long n_joints,
                      float gscale, void* stream);

/* Joint-angle loss (train_mixer_h36m.py:187, train_autoreg_mixer_h36m.py:209-210): mean over the rows of sum_d |pred - gt|.
 * *loss_sum += sum |pred - gt| (caller zeroes it; mean = loss_sum / rows); dpred (nullable) = gscale * sign(pred - gt) / rows. */
int mmx_l1_fwd_bwd(const float* pred, const float* gt, float* dpred, float* loss_sum, long long rows, int D, float gscale, void* stream);

/* torch.optim.Adam (coupled L2) on flat buffers — train_mixer_h36m.py:63,193.
 * hyper (DEVICE, 10 floats): lr, beta1, beta2, eps, weight_decay, 1-beta1^t, sqrt(1-beta2^t), grad_scale,
 * 1-beta1, 1-beta2 (the last two rounded once from double, as PyTorch does). */
int mmx_adam_step(float* p, const float* g, float* m, float* v, long long n, const float* hyper, void* stream);
/* Device-side optimiser clock: ++*step (DEVICE uint32, also the dropout step_dev); hyper[5], hyper[6] are
 * recomputed from hyper[1], hyper[2] and the new step.  Lets a CUDA graph replay a whole training step. */
int mmx_adam_advance(float* hyper, unsigned int* step, void* stream);

/* ---------------- data parallelism: gradient exchange fused into the optimiser (one process per GPU, one node) ----------------
 * The reference trains on one device; the north star asks for batch-sharded data parallelism with one bucketed gradient
 * all-reduce.  mmx_adam_step_peer is that all-reduce AND mmx_adam_step in one kernel over NVLink peer memory: every rank's flat
 * gradient bucket lives in an allocation made by mmx_peer_alloc (cudaMalloc, zeroed; bucket first, then mmx_peer_flag_bytes(world)
 * bytes of flags), exported with mmx_ipc_export (64-byte cudaIpcMemHandle_t), exchanged by the caller (torch.distributed) and
 * mapped by every peer with mmx_ipc_open.  peer_g / peer_flags: DEVICE arrays [world] of the bucket / flag-block addresses of
 * every rank as mapped in THIS process (own rank: the local pointer).  Sums in rank order on every rank (replicas stay
 * bit-identical); hyper as mmx_adam_step (hyper[7] = 1/world); epoch: DEVICE uint32[2], zero-initialised, owned by the kernel.
 * Collective: every rank must launch it the same number of times.  Waits are bounded (~15 s; then mmx_tc5_abort_count() > 0). */
int mmx_peer_flag_bytes(int world);
int mmx_peer_alloc(long long bytes, void** ptr);
int mmx_peer_free(void* ptr);
int mmx_ipc_export(void* ptr, unsigned char* handle64);
int mmx_ipc_open(const unsigned char* handle64, void** ptr);
int mmx_ipc_close(void* ptr);
int mmx_adam_step_peer(float* p, float* m, float* v, const void* peer_g, const void* peer_flags, int rank, int world, long long n,
                       const float* hyper, unsigned int* epoch, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MMX_H_ */
