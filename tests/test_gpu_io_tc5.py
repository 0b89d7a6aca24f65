"""The tcgen05 embedding and output head of the MlpMixer (precision "tf32") against an fp64 reference, kernel by kernel.

  * csrc/mmx_lin_tc5.cuh: the row-wise linear layer y = x W^T + b (MlpMixer.conv), mmx_linear_{fwd,bwd}_prec.  Two plans:
    operand width 64 when max(K+1, N) <= 64, else 80.
  * csrc/mmx_head_tc5.cuh: the whole head fc_out(conv_out(LN(x))) as one kernel per direction, mmx_mlp_head_{fwd,bwd}_prec.
    A tile is S = 128 / max(T, To) whole sequences; the time-mix weight gradient accumulates in TMEM over a CTA's tiles.

Bar: 2e-4 relative per tensor (max|got-want| <= 2e-4 max|want|).  Derived, not measured: the bf16 hi+lo split leaves about
2^-16 per product (the headers claim ~1e-5 overall), so 2e-4 keeps a 10x margin; a product that drops one cross term (lo*hi)
is off by about 2^-9 = 2e-3, the model bar, which therefore cannot see it.

Every served case checks, besides the values:
  * the tcgen05 kernel ran: the tf32 result differs from the fp32 one (0 < d < bar), and with MMX_IO_NO_TC5=1 the tf32 call
    gives the fp32 result (outputs bit for bit; accumulated gradients up to the order of the fp32 kernels' atomics);
  * nothing is written past the end: every output has a NaN canary tail of one tile, which must stay NaN bit for bit;
  * gradients accumulate: the buffers start at known nonzero values G0 and got - G0 is compared;
  * a sparse upstream gradient (~64 rows / sequences, the first and the last included) leaves dx exactly 0 elsewhere, and the
    weight gradients equal those of the selected rows alone: a tile that reads another tile's data, or a flush that reads the
    wrong block of the (block-diagonal) time-mix gradient, shows up there;
  * mmx_tc5_abort_count() does not move.
Shapes the tcgen05 kernels decline must give the fp32 result bit for bit and match the reference to 1e-5.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import mixer_np as O
from tests.golden_util import check_close

BAR = 2e-4          # tcgen05 kernels, every tensor
BAR_FP32 = 1e-5     # fp32 kernels (the fall-back cases)
ATOMIC_ORDER = 1e-5  # fp32 gradients summed by atomics from several CTAs: the order varies (measured up to 2.4e-6)
N_SPARSE = 64
FP32, TF32 = 0, 1
MMX_E_UNSUPPORTED = -2


# ------------------------------------------------------------------------------------------ fp64 references
def lin_fwd_ref(x, w, b):
    return x @ w.T + b


def lin_bwd_ref(x, w, dy):
    """dW, db, dx of y = x W^T + b."""
    return dy.T @ x, dy.sum(0), dy @ w


def head_fwd_ref(x, p):
    """x [B,T,H]; p = (ln_w [H], ln_b [H], wt [To,T,1], bt [To], wf [D,H], bf [D]).  Returns out [B,To,D] and what the
    backward needs."""
    ln_w, ln_b, wt, bt, wf, bf = p
    z, ln_cache = O.ln_fwd(x, ln_w, ln_b)
    P = np.matmul(wt[:, :, 0], z) + bt[None, :, None]           # conv_out over the frames
    return P @ wf.T + bf, (z, ln_cache, P)


def head_bwd_ref(p, saved, dout):
    """dx and the gradients of (ln_w, ln_b, wt, bt, wf, bf)."""
    ln_w, _, wt, _, wf, _ = p
    z, ln_cache, P = saved
    D, H = wf.shape
    g_wf = dout.reshape(-1, D).T @ P.reshape(-1, H)
    g_bf = dout.reshape(-1, D).sum(0)
    dP = dout @ wf
    g_wt = np.tensordot(dP, z, axes=([0, 2], [0, 2]))[:, :, None]
    g_bt = dP.sum((0, 2))
    dx, g_lnw, g_lnb = O.ln_bwd(np.matmul(wt[:, :, 0].T, dP), ln_cache, ln_w)
    return dx, [g_lnw, g_lnb, g_wt, g_bt, g_wf, g_bf]


HEAD_PARAM_NAMES = ("ln_w", "ln_b", "wt", "bt", "wf", "bf")


def lin_data(R, K, N, seed):
    rng = np.random.default_rng(seed)
    x = (3.0 + rng.standard_normal((R, K))).astype(np.float32)
    w = (rng.standard_normal((N, K)) / np.sqrt(K)).astype(np.float32)
    b = (0.3 * rng.standard_normal(N)).astype(np.float32)
    dy = rng.standard_normal((R, N)).astype(np.float32)
    return x, w, b, dy


def head_data(B, T, To, H, D, seed):
    rng = np.random.default_rng(seed)
    x = (3.0 + rng.standard_normal((B, T, H))).astype(np.float32)     # the mean offset exercises the shifted LN statistics
    p = [1.0 + 0.3 * rng.standard_normal(H), 0.3 * rng.standard_normal(H), rng.standard_normal((To, T, 1)) / np.sqrt(T),
         0.3 * rng.standard_normal(To), rng.standard_normal((D, H)) / np.sqrt(H), 0.3 * rng.standard_normal(D)]
    dout = rng.standard_normal((B, To, D)).astype(np.float32)
    return x, [q.astype(np.float32) for q in p], dout


def sparse_rows(n_rows, seed, n=N_SPARSE):
    """The first and the last row and a seeded sample spread over the rest."""
    rng = np.random.default_rng(seed)
    mid = rng.choice(np.arange(1, n_rows - 1), size=min(n, n_rows) - 2, replace=False) if n_rows > 2 else []
    return np.unique(np.concatenate([[0, n_rows - 1], mid])).astype(np.int64)


def test_references_match_float64_autograd():
    """The hand-written fp64 backward above against torch.float64 autograd of the same formulas (CPU)."""
    for R, K, N in [(7, 8, 8), (37, 66, 50), (20, 50, 66)]:
        x, w, b, dy = (a.astype(np.float64) for a in lin_data(R, K, N, seed=R))
        xt, wt_, bt_ = (torch.from_numpy(a).requires_grad_(True) for a in (x, w, b))
        y = torch.nn.functional.linear(xt, wt_, bt_)
        y.backward(torch.from_numpy(dy))
        np.testing.assert_allclose(lin_fwd_ref(x, w, b), y.detach().numpy(), rtol=1e-12, atol=1e-12)
        for got, want in zip(lin_bwd_ref(x, w, dy), (wt_.grad, bt_.grad, xt.grad)):
            np.testing.assert_allclose(got, want.numpy(), rtol=1e-12, atol=1e-11)
    for B, T, To, H, D in [(3, 10, 10, 50, 66), (4, 10, 25, 50, 54), (5, 25, 10, 48, 12), (2, 40, 7, 8, 8), (6, 1, 1, 8, 8)]:
        x, p, dout = head_data(B, T, To, H, D, seed=B * T)
        x, dout, p = x.astype(np.float64), dout.astype(np.float64), [q.astype(np.float64) for q in p]
        out, saved = head_fwd_ref(x, p)
        dx, grads = head_bwd_ref(p, saved, dout)
        xt = torch.from_numpy(x).requires_grad_(True)
        pt = [torch.from_numpy(q).requires_grad_(True) for q in p]
        z = torch.nn.functional.layer_norm(xt, (H,), pt[0], pt[1], 1e-5)
        P = torch.nn.functional.conv1d(z, pt[2], pt[3])              # Conv1d(seq_len, pred_len, 1): frames are the channels
        ot = torch.nn.functional.linear(P, pt[4], pt[5])
        ot.backward(torch.from_numpy(dout))
        np.testing.assert_allclose(out, ot.detach().numpy(), rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(dx, xt.grad.numpy(), rtol=1e-10, atol=1e-11)
        for name, got, q in zip(HEAD_PARAM_NAMES, grads, pt):
            np.testing.assert_allclose(got, q.grad.numpy(), rtol=1e-10, atol=1e-10, err_msg=name)


# ------------------------------------------------------------------------------------------ device plumbing
def _lib():
    from motionmixerconv_b200 import _lib as L
    return L, L.load()


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _dev(a, offset=0):
    """a on the device; offset > 0 gives a view that starts `offset` floats into its buffer (misaligned for offset 1)."""
    buf = torch.empty(a.size + offset, dtype=torch.float32, device="cuda")
    t = buf[offset:].view(a.shape)
    t.copy_(torch.from_numpy(np.ascontiguousarray(a)))
    return t


class Out:
    """An output buffer the kernel gets a view of: `canary` floats of NaN follow it, and it starts at g0 (gradients) or NaN."""

    def __init__(self, shape, canary, g0=None, offset=0):
        self.n = int(np.prod(shape))
        self.buf = torch.full((offset + self.n + canary,), float("nan"), device="cuda")
        self.t = self.buf[offset:offset + self.n].view(shape)
        self.g0 = g0
        if g0 is not None:
            self.t.copy_(torch.from_numpy(g0))
        self.offset = offset
        self.canary = self.buf[offset + self.n:].view(torch.int32).clone()

    @property
    def ptr(self):
        return self.t.data_ptr()

    def get(self, what):
        """The result (minus g0); asserts that the canary tail is untouched."""
        torch.cuda.synchronize()
        assert torch.equal(self.buf[self.offset + self.n:].view(torch.int32), self.canary), "%s: written past its end" % what
        got = self.t.cpu().numpy()
        return got if self.g0 is None else got.astype(np.float64) - self.g0


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max()) / max(float(np.abs(b).max()), 1e-30)


def _check_route(run, monkeypatch, exact, fp32_served=True):
    """run(precision) -> dict of results.  Asserts that the tf32 call ran the tcgen05 kernel (it differs from fp32 by
    0 < d < BAR in the first result) and that MMX_IO_NO_TC5=1 turns it into the fp32 call: bit for bit for the names in
    `exact`, within ATOMIC_ORDER for accumulated gradients.  fp32_served=False: the fp32 kernels decline the shape
    (MMX_E_UNSUPPORTED), so the tf32 call must too once tcgen05 is switched off.  Returns the tf32 results."""
    got = run(TF32)
    assert isinstance(got, dict), "the tf32 call failed with %r" % (got,)
    if fp32_served:
        ref = run(FP32)
        k0 = next(iter(got))
        d = _rel(got[k0], ref[k0])
        assert 0.0 < d < BAR, (k0, d)
    else:
        assert run(FP32) == MMX_E_UNSUPPORTED
    monkeypatch.setenv("MMX_IO_NO_TC5", "1")
    try:
        off = run(TF32)
    finally:
        monkeypatch.delenv("MMX_IO_NO_TC5")
    if not fp32_served:
        assert off == MMX_E_UNSUPPORTED
        return got
    for k in got:
        if k in exact:
            assert np.array_equal(off[k], ref[k]), "%s: MMX_IO_NO_TC5=1 differs from fp32" % k
        else:
            assert _rel(off[k], ref[k]) <= ATOMIC_ORDER, k
    return got


# ------------------------------------------------------------------------------------------ linear layer
def lin_fwd(x, w, b, prec, y_off=0):
    L, lib = _lib()
    R, K = x.shape
    N = w.shape[0]
    y = Out((R, N), 128 * N, offset=y_off)
    L.check(lib, lib.mmx_linear_fwd_prec(R, K, N, x.data_ptr(), w.data_ptr(), b.data_ptr(), y.ptr, prec, _stream()), "mmx_linear_fwd_prec")
    return {"y": y.get("y")}


def lin_bwd(x, w, dy, prec, want_dx, g0, dx_off=0):
    L, lib = _lib()
    R, K = x.shape
    N = w.shape[0]
    dw, db = Out((N, K), 64, g0[0]), Out((N,), 64, g0[1])
    dx = Out((R, K), 128 * K, offset=dx_off) if want_dx else None
    rc = lib.mmx_linear_bwd_prec(R, K, N, x.data_ptr(), w.data_ptr(), dy.data_ptr(), dw.ptr, db.ptr, dx.ptr if want_dx else None, prec, _stream())
    L.check(lib, rc, "mmx_linear_bwd_prec")
    out = {"dw": dw.get("dw"), "db": db.get("db")}
    if want_dx:
        out["dx"] = dx.get("dx")
    return out


LIN_SHAPES = [
    (8, 8), (54, 50), (62, 64), (50, 62),        # operand width 64 at its edges (K+1 = 63, N = 64)
    (64, 50),                                    # K+1 = 65: the first shape of the width-80 plan
    (66, 50),                                    # the embedding of the headline model
    (50, 66),                                    # fc_out-like
    (78, 80),                                    # width 80 at its edges (K+1 = 79, N = 80)
]


def lin_rows(kind):
    """One full tile; one ragged tile; >= 3 tiles per CTA (grid <= 2 x SMs) with a ragged last tile.  rows*K stays a
    multiple of 4 for every even K."""
    return {"tile": 128, "ragged": 100, "multi": 6 * _sms() * 128 + 74}[kind]


@pytest.mark.gpu
@pytest.mark.parametrize("rows", ["tile", "ragged", "multi"])
@pytest.mark.parametrize("K,N", LIN_SHAPES, ids=["K%d_N%d" % s for s in LIN_SHAPES])
def test_linear_vs_fp64(K, N, rows, monkeypatch):
    L, lib = _lib()
    abort0 = lib.mmx_tc5_abort_count()
    R = lin_rows(rows)
    assert R * K % 4 == 0
    x, w, b, dy = lin_data(R, K, N, seed=[K, N, R])
    x64, w64 = x.astype(np.float64), w.astype(np.float64)
    xd, wd, bd, dyd = _dev(x), _dev(w), _dev(b), _dev(dy)
    rng = np.random.default_rng(1)
    g0 = [(1.0 + rng.standard_normal(s)).astype(np.float32) for s in ((N, K), (N,))]

    got = _check_route(lambda p: lin_fwd(xd, wd, bd, p), monkeypatch, exact={"y"})
    check_close("y", got["y"], lin_fwd_ref(x64, w64, b), rtol=BAR)

    want = dict(zip(("dw", "db", "dx"), lin_bwd_ref(x64, w64, dy.astype(np.float64))))
    for want_dx in (True, False):
        got = _check_route(lambda p: lin_bwd(xd, wd, dyd, p, want_dx, g0), monkeypatch, exact={"dx"})
        assert set(got) == ({"dw", "db", "dx"} if want_dx else {"dw", "db"})
        for k, v in got.items():
            check_close(k, v, want[k], rtol=BAR)

    # sparse upstream gradient
    q = sparse_rows(R, seed=R)
    dys = np.zeros_like(dy)
    dys[q] = dy[q]
    got = lin_bwd(xd, wd, _dev(dys), TF32, True, g0)
    rest = np.ones(R, bool)
    rest[q] = False
    assert not got["dx"][rest].any(), "dx nonzero outside the rows that carry dy"
    dws, dbs, dxs = lin_bwd_ref(x64[q], w64, dys[q].astype(np.float64))
    check_close("dw (sparse dy)", got["dw"], dws, rtol=BAR)
    check_close("db (sparse dy)", got["db"], dbs, rtol=BAR)
    check_close("dx (sparse dy)", got["dx"][q], dxs, rtol=BAR)
    assert lib.mmx_tc5_abort_count() == abort0


LIN_FALLBACK = {
    "K80": dict(R=1000, K=80, N=50),              # K+1 > 80
    "N82": dict(R=1000, K=50, N=82),
    "K_odd": dict(R=128, K=55, N=50),
    "rowsK_not4": dict(R=129, K=54, N=50),        # rows*K % 4 != 0: a tile is not a whole number of 16-byte units
    "x_off4": dict(R=1000, K=66, N=50, x_off=1),  # pointers 4 bytes off 16-byte alignment
    "y_off4": dict(R=1000, K=66, N=50, y_off=1),  # y in the forward, dy in the backward
    "dx_off4": dict(R=1000, K=66, N=50, dx_off=1),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(LIN_FALLBACK))
def test_linear_declined_shapes_give_the_fp32_result(name):
    c = {"x_off": 0, "y_off": 0, "dx_off": 0, **LIN_FALLBACK[name]}
    R, K, N = c["R"], c["K"], c["N"]
    x, w, b, dy = lin_data(R, K, N, seed=[K, N, R])
    x64, w64 = x.astype(np.float64), w.astype(np.float64)
    xd, wd, bd, dyd = _dev(x, c["x_off"]), _dev(w), _dev(b), _dev(dy, c["y_off"])
    g0 = [np.full((N, K), 0.5, np.float32), np.full(N, -0.25, np.float32)]
    yt, yf = (lin_fwd(xd, wd, bd, p, y_off=c["y_off"]) for p in (TF32, FP32))
    if c["dx_off"]:                 # dx is a backward-only tensor: the forward stays on tcgen05
        assert 0.0 < _rel(yt["y"], yf["y"]) < BAR
        check_close("y", yt["y"], lin_fwd_ref(x64, w64, b), rtol=BAR)
    else:
        assert np.array_equal(yt["y"], yf["y"])
        check_close("y", yt["y"], lin_fwd_ref(x64, w64, b), rtol=BAR_FP32)
    gt, gf = (lin_bwd(xd, wd, dyd, p, True, g0, dx_off=c["dx_off"]) for p in (TF32, FP32))
    assert np.array_equal(gt["dx"], gf["dx"])
    want = dict(zip(("dw", "db", "dx"), lin_bwd_ref(x64, w64, dy.astype(np.float64))))
    for k in ("dw", "db", "dx"):
        assert _rel(gt[k], gf[k]) <= ATOMIC_ORDER, k
        check_close(k, gt[k], want[k], rtol=BAR_FP32)


# ------------------------------------------------------------------------------------------ output head
def _head_tables(params):
    from motionmixerconv_b200 import functional as F_
    return F_.mlp_head_table(params)


def head_fwd(dims, x, params, prec, S):
    """dims = (B, T, To, H, D).  Returns the results, or the return code when the call fails."""
    L, lib = _lib()
    B, T, To, H, D = dims
    out = Out((B, To, D), S * To * D)
    rc = lib.mmx_mlp_head_fwd_prec(C.byref(L.MmxMlpHeadDesc(*dims)), C.byref(_head_tables(params)), x.data_ptr(), out.ptr, prec, _stream())
    if rc != 0:
        return rc
    return {"out": out.get("out")}


def head_bwd(dims, x, params, dout, prec, S, g0):
    L, lib = _lib()
    B, T, To, H, D = dims
    dx = Out((B, T, H), S * T * H)
    grads = [Out(g.shape, 64, g) for g in g0]
    rc = lib.mmx_mlp_head_bwd_prec(C.byref(L.MmxMlpHeadDesc(*dims)), C.byref(_head_tables(params)), C.byref(_head_tables([g.t for g in grads])),
                                   x.data_ptr(), dout.data_ptr(), dx.ptr, prec, _stream())
    if rc != 0:
        return rc
    res = {"dx": dx.get("dx")}
    for n, g in zip(HEAD_PARAM_NAMES, grads):
        res["g_" + n] = g.get("g_" + n)
    return res


HEAD_SHAPES = {                    # (T, To, H, D)
    "T10_To10_H50_D66": (10, 10, 50, 66),        # headline
    "T10_To24_H50_D54": (10, 24, 50, 54),        # D = 54 (AMASS), To > T, S = 5
    "T25_To10_H48_D12": (25, 10, 48, 12),        # T > To
    "T16_To16_H62_D80": (16, 16, 62, 80),        # H + 1 = 63 of KH = 64, D = KD = 80
    "T1_To1_H8_D8": (1, 1, 8, 8),                # S = 128: full 128-row tiles
    "T11_To13_H44_D20": (11, 13, 44, 20),        # odd S*T and S*To
    "T40_To10_H50_D66": (40, 10, 50, 66),        # T > 32: the fp32 kernels do not serve these
    "T100_To7_H48_D12": (100, 7, 48, 12),        # S = 1
    "T128_To128_H8_D8": (128, 128, 8, 8),        # the largest T, To
}


def head_batch(kind, T, To):
    """A small batch with a ragged second tile, or B = 3 x SMs x S + r: CTA 0 runs 4 tiles (grid <= SMs), the last ragged."""
    S = 128 // max(T, To)
    r = (S + 1) // 2 if S > 1 else 1
    return S, (S + r if kind == "ragged" else 3 * _sms() * S + r)


@pytest.mark.gpu
@pytest.mark.parametrize("batch", ["ragged", "multi"])
@pytest.mark.parametrize("name", list(HEAD_SHAPES))
def test_head_vs_fp64(name, batch, monkeypatch):
    L, lib = _lib()
    abort0 = lib.mmx_tc5_abort_count()
    T, To, H, D = HEAD_SHAPES[name]
    S, B = head_batch(batch, T, To)
    dims = (B, T, To, H, D)
    x, p, dout = head_data(B, T, To, H, D, seed=[B, T, To, H, D])
    x64, p64 = x.astype(np.float64), [q.astype(np.float64) for q in p]
    xd, pd, doutd = _dev(x), [_dev(q) for q in p], _dev(dout)
    rng = np.random.default_rng(2)
    g0 = [(1.0 + rng.standard_normal(q.shape)).astype(np.float32) for q in p]
    fp32_served = T <= 32

    out64, saved = head_fwd_ref(x64, p64)
    got = _check_route(lambda pr: head_fwd(dims, xd, pd, pr, S), monkeypatch, exact={"out"}, fp32_served=fp32_served)
    check_close("out", got["out"], out64, rtol=BAR)

    dx64, g64 = head_bwd_ref(p64, saved, dout.astype(np.float64))
    want = dict(dx=dx64, **{"g_" + n: g for n, g in zip(HEAD_PARAM_NAMES, g64)})
    got = _check_route(lambda pr: head_bwd(dims, xd, pd, doutd, pr, S, g0), monkeypatch, exact={"dx"}, fp32_served=fp32_served)
    for k, v in got.items():
        check_close(k, v, want[k], rtol=BAR)

    # sparse upstream gradient: whole sequences
    q = sparse_rows(B, seed=B)
    douts = np.zeros_like(dout)
    douts[q] = dout[q]
    got = head_bwd(dims, xd, pd, _dev(douts), TF32, S, g0)
    rest = np.ones(B, bool)
    rest[q] = False
    assert not got["dx"][rest].any(), "dx nonzero outside the sequences that carry dout"
    _, saved_q = head_fwd_ref(x64[q], p64)
    dxq, gq = head_bwd_ref(p64, saved_q, douts[q].astype(np.float64))
    check_close("dx (sparse dout)", got["dx"][q], dxq, rtol=BAR)
    for n, g in zip(HEAD_PARAM_NAMES, gq):
        check_close("g_%s (sparse dout)" % n, got["g_" + n], g, rtol=BAR)
    assert lib.mmx_tc5_abort_count() == abort0


HEAD_FALLBACK = {                  # (T, To, H, D, x offset in floats)
    "H64": (10, 10, 64, 66, 0),                 # H + 1 > KH
    "H63": (12, 12, 63, 66, 0),                 # odd H (T*H % 4 == 0)
    "D82": (10, 10, 50, 82, 0),                 # D > KD
    "TH_not4": (11, 10, 50, 66, 0),             # T*H % 4 != 0
    "ToD_not4": (10, 25, 50, 54, 0),            # To*D % 4 != 0: the AMASS head (pred_len 25, 54 outputs)
    "x_off4": (10, 10, 50, 66, 1),              # x 4 bytes off 16-byte alignment
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(HEAD_FALLBACK))
def test_head_declined_shapes_give_the_fp32_result(name):
    T, To, H, D, off = HEAD_FALLBACK[name]
    B = 333
    dims = (B, T, To, H, D)
    x, p, dout = head_data(B, T, To, H, D, seed=[B, T, To, H, D])
    x64, p64 = x.astype(np.float64), [q.astype(np.float64) for q in p]
    xd, pd, doutd = _dev(x, off), [_dev(q) for q in p], _dev(dout)
    g0 = [np.full(q.shape, 0.5, np.float32) for q in p]
    ot, of = (head_fwd(dims, xd, pd, pr, 1) for pr in (TF32, FP32))
    assert np.array_equal(ot["out"], of["out"])
    out64, saved = head_fwd_ref(x64, p64)
    check_close("out", ot["out"], out64, rtol=BAR_FP32)
    gt, gf = (head_bwd(dims, xd, pd, doutd, pr, 1, g0) for pr in (TF32, FP32))
    assert np.array_equal(gt["dx"], gf["dx"])
    dx64, g64 = head_bwd_ref(p64, saved, dout.astype(np.float64))
    want = dict(dx=dx64, **{"g_" + n: g for n, g in zip(HEAD_PARAM_NAMES, g64)})
    for k in want:
        assert _rel(gt[k], gf[k]) <= ATOMIC_ORDER, k
        check_close(k, gt[k], want[k], rtol=BAR_FP32)


@pytest.mark.gpu
def test_fp32_head_still_declines_T_above_32():
    """Only the tcgen05 head serves T > 32: the fp32 mode, and tf32 on a shape tcgen05 declines (odd H), give
    MMX_E_UNSUPPORTED as before."""
    for (T, To, H, D), prec in [((40, 10, 50, 66), FP32), ((33, 10, 50, 66), FP32), ((40, 10, 51, 66), TF32), ((40, 10, 64, 66), TF32)]:
        B = 5
        x, p, dout = head_data(B, T, To, H, D, seed=1)
        xd, pd, doutd = _dev(x), [_dev(q) for q in p], _dev(dout)
        g0 = [np.zeros(q.shape, np.float32) for q in p]
        assert head_fwd((B, T, To, H, D), xd, pd, prec, 1) == MMX_E_UNSUPPORTED
        assert head_bwd((B, T, To, H, D), xd, pd, doutd, prec, 1, g0) == MMX_E_UNSUPPORTED


# ------------------------------------------------------------------------------------------ whole model
MODEL_VARIANTS = {
    # AMASS-shaped: embedding K+1 = 55, N = 50 on the width-64 plan; the head (To*D = 1350) falls back to fp32
    "amass_h50_to25": dict(input_size=54, num_classes=54, hidden_dim=50, channels_mlp_dim=50, pred_len=25),
    # embedding N = 64 on the width-64 plan; the head (H + 1 = 65 > 64) falls back to fp32
    "amass_h64": dict(input_size=54, num_classes=54, hidden_dim=64, channels_mlp_dim=64),
    # embedding K+1 = 79 on the width-80 plan; the head at H + 1 = 63, D = 78
    "h62_d78": dict(input_size=78, num_classes=78, hidden_dim=62, channels_mlp_dim=62),
}


@pytest.mark.gpu
@pytest.mark.parametrize("batch", ["b515", "multi"])
@pytest.mark.parametrize("name", sorted(MODEL_VARIANTS))
def test_model_variants_vs_oracle(name, batch, monkeypatch):
    from tests.golden_util import Golden
    from tests.synthetic import synthetic_pose_windows
    from tests.test_gpu_mlp_tc5 import _compare, _model, _oracle, _run
    L, lib = _lib()
    abort0 = lib.mmx_tc5_abort_count()
    cfg = dict(Golden("mlp_k2").cfg, num_blocks=2, regularization=0, **MODEL_VARIANTS[name])
    T, To, D = cfg["seq_len"], cfg["pred_len"], cfg["input_size"]
    B = 515 if batch == "b515" else head_batch("multi", T, To)[1]
    model = _model(cfg, None, seed=3).train()
    params = {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}
    x, gt = synthetic_pose_windows(B, T, To, D, scale="amass", seed=9)
    _compare(*_run(model, x, gt), _oracle(cfg, params, x, gt))
    xd = torch.from_numpy(x).cuda()
    with torch.no_grad():
        a = model(xd)
        monkeypatch.setenv("MMX_IO_NO_TC5", "1")
        b = model(xd)
        monkeypatch.delenv("MMX_IO_NO_TC5")
    d = (a - b).abs().max().item() / b.abs().max().item()
    assert 0.0 < d < 2e-3, d                     # the tcgen05 embedding / head served it
    assert lib.mmx_tc5_abort_count() == abort0
