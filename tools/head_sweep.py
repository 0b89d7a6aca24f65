import ctypes as C, os, sys, json
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from motionmixerconv_b200 import _lib as L
from motionmixerconv_b200 import functional as F_
lib = L.load()
B, T, To, H, D = 4096, 10, 25, 128, 54
x = torch.randn(B, T, H, device="cuda"); dout = torch.randn(B, To, D, device="cuda")
out = torch.empty(B, To, D, device="cuda"); dx = torch.empty_like(x)
ps = [torch.randn(H, device="cuda"), torch.randn(H, device="cuda"), torch.randn(To, T, 1, device="cuda") * .3, torch.randn(To, device="cuda"),
      torch.randn(D, H, device="cuda") * .1, torch.randn(D, device="cuda")]
gs = [torch.zeros_like(p) for p in ps]
w, g = F_.mlp_head_table(ps), F_.mlp_head_table(gs)
desc = L.MmxMlpHeadDesc(B, T, To, H, D)
st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
def t(fn, n=20):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(n): fn()
    e.record(); torch.cuda.synchronize()
    return s.elapsed_time(e) / n * 1e3
f = t(lambda: L.check(lib, lib.mmx_mlp_head_fwd(C.byref(desc), C.byref(w), x.data_ptr(), out.data_ptr(), st), "f"))
b = t(lambda: L.check(lib, lib.mmx_mlp_head_bwd(C.byref(desc), C.byref(w), C.byref(g), x.data_ptr(), dout.data_ptr(), dx.data_ptr(), st), "b"))
print(json.dumps({"S_fwd": os.environ.get("MMX_HEAD_S_FWD"), "S_bwd": os.environ.get("MMX_HEAD_S_BWD"), "fwd_us": round(f, 1), "bwd_us": round(b, 1)}))
