"""LayerNorm kernel device time at the BASELINE stage shapes (run on the GPU box): raw C-ABI calls captured in a CUDA
graph (20 launches per replay, rotating buffers larger than L2)."""
import ctypes as C, json, os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pwa_b200
from pwa_b200 import _lib
from pwa_b200.functional import _ptr, _stream

dev = torch.device("cuda")
NB = 6
def graph_time(fn, reps=20):
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        for i in range(3): fn(i)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(reps): fn(i)
    g.replay(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); g.replay(); g.replay(); e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (2 * reps) * 1e3

for rows, Cc in ((4 * 432 * 256, 48), (4 * 54 * 256, 96), (4 * 28 * 256, 192), (4 * 13824, 384), (4 * 1728, 768)):
    dt = torch.bfloat16
    mk = lambda: [torch.randn(rows, Cc, device=dev).to(dt) for _ in range(NB)]
    x, r, s_, y, dy, dx = mk(), mk(), mk(), mk(), mk(), mk()
    g, b = torch.randn(Cc, device=dev), torch.randn(Cc, device=dev)
    mean, rstd = torch.empty(rows, device=dev), torch.empty(rows, device=dev)
    dg, db, c1, c2 = (torch.empty(Cc, device=dev) for _ in range(4))
    L = _lib.lib
    def fwd(i):
        i %= NB
        _lib.check(L.pwa_ln_fwd(_ptr(x[i]), None, _ptr(g), _ptr(b), None, _ptr(y[i]), _ptr(mean), _ptr(rstd), rows, Cc, 1e-6, 1, _stream(g)), "f")
    def fwd_res(i):
        i %= NB
        _lib.check(L.pwa_ln_fwd(_ptr(x[i]), _ptr(r[i]), _ptr(g), _ptr(b), _ptr(s_[i]), _ptr(y[i]), _ptr(mean), _ptr(rstd), rows, Cc, 1e-6, 1, _stream(g)), "fr")
    def bwd(i):
        i %= NB
        _lib.check(L.pwa_ln_bwd2(_ptr(dy[i]), _ptr(x[i]), _ptr(g), _ptr(mean), _ptr(rstd), None, _ptr(dx[i]), _ptr(dg), _ptr(db), None, None, rows, Cc, 1, _stream(g)), "b")
    def bwd_res(i):
        i %= NB
        _lib.check(L.pwa_ln_bwd2(_ptr(dy[i]), _ptr(x[i]), _ptr(g), _ptr(mean), _ptr(rstd), _ptr(r[i]), _ptr(dx[i]), _ptr(dg), _ptr(db), _ptr(c1), _ptr(c2), rows, Cc, 1, _stream(g)), "br")
    fwd(0); torch.cuda.synchronize()
    nb = rows * Cc * 2
    t = [graph_time(f) for f in (fwd, fwd_res, bwd, bwd_res)]
    print(json.dumps({"rows": rows, "C": Cc, "fwd_us": round(t[0], 1), "fwd_GBs": round(2 * nb / t[0] / 1e3),
                      "fwd_res_us": round(t[1], 1), "fwd_res_GBs": round(4 * nb / t[1] / 1e3), "bwd_us": round(t[2], 1),
                      "bwd_GBs": round(3 * nb / t[2] / 1e3), "bwd_res_us": round(t[3], 1), "bwd_res_GBs": round(4 * nb / t[3] / 1e3)}))
