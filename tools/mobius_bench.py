import ctypes as C, sys, os
sys.path.insert(0, os.path.join(os.path.dirname(__file__), ".."))
import torch
from multilinear_b200 import api as ml
from multilinear_b200 import load
L = load(); ml.set_device(0)
for nv in (20, 22, 24):
    n = 1 << nv
    ev = ml.synthetic_elements_dev(1, n); out = ml.DeviceBuffer(16 * n)
    f = lambda: ml.check(L.ml_mle_to_coefficient_dev(ev.ptr, C.c_size_t(n), out.ptr, None))
    for _ in range(3): f()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20): f()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 20
    print("mobius 2^%d: %.4f ms  %.0f GB/s alg" % (nv, ms, 32 * n / ms / 1e6))
