"""Experiment: screen kernel time, top-1 vs top-k, by shape / k (diagnostic)."""
import os, sys, ctypes
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from video_similarity_search_b200 import _lib
from video_similarity_search_b200.backend import CudaBackend
be = CudaBackend(); lib = _lib.load()
def mixture(m, d, kc, g, centres):
    out = torch.empty(m, d, device="cuda")
    for s in range(0, m, 65536):
        e = min(m, s + 65536)
        lab = torch.randint(0, kc, (e - s,), device="cuda", generator=g)
        out[s:e] = centres[lab] + torch.randn(e - s, d, device="cuda", generator=g)
    return out
TRACE = os.environ.get("TRACE", "0") == "1"
def screen_ms(fn):
    fn(); torch.cuda.synchronize()
    lib.slic_profile_screen(1)
    fn(); torch.cuda.synchronize()
    ms = ctypes.c_float(0); fl = ctypes.c_double(0)
    lib.slic_last_screen_time(ctypes.byref(ms), ctypes.byref(fl))
    lib.slic_profile_screen(0)
    if TRACE:
        lib.slic_screen_trace(1, None)
        fn(); torch.cuda.synchronize()
        c = (ctypes.c_uint64 * 12)()
        lib.slic_screen_trace(0, c)
        c = [v / 148.0 / 1e6 for v in c]
        print("    trace (Mcycles per CTA): producer-wait %.2f | mma: wait-acc %.2f wait-operands %.2f total %.2f | epi0: wait-mma %.2f total %.2f | chunks triggered %.3f of %.3f M"
              % tuple(c[:8]))
    return ms.value, fl.value / ms.value / 1e9
for shape in sys.argv[1:]:
    nq, n, d = [int(v) for v in shape.split("x")]
    kc = max(2, n // 1000)
    g = torch.Generator(device="cuda").manual_seed(0)
    centres = torch.randn(kc, d, device="cuda", generator=g)
    x, q = mixture(n, d, kc, g, centres), mixture(nq, d, kc, g, centres)
    ux, xb = be.normalize_rows(x); uq, qb = be.normalize_rows(q)
    ms, tf = screen_ms(lambda: be.nn_top1(uq, qb, ux, xb))
    print("%s top1: %.3f ms %.0f TF/s" % (shape, ms, tf), flush=True)
    for k in (1, 20, 50):
        ms, tf = screen_ms(lambda: be.topk_cosine(uq, ux, k, q_f16=qb, x_f16=xb))
        st = be.last_stats.cpu().tolist()
        print("%s top%d: %.3f ms %.0f TF/s  reranked/row %.0f listed/row %.0f compactions %d" % (shape, k, ms, tf, st[0] / nq, st[3] * 16.0 / nq, st[2]), flush=True)
