import ctypes as C, os, sys
sys.path.insert(0, os.path.join(os.path.dirname(__file__), ".."))
from multilinear_b200 import api as ml
from multilinear_b200 import load
L = load(); ml.set_device(0)
n = 1 << 24
ev = ml.synthetic_elements_dev(1, n); out = ml.DeviceBuffer(16 * n)
for _ in range(2): ml.check(L.ml_mle_to_coefficient_dev(ev.ptr, C.c_size_t(n), out.ptr, None))
ml.synchronize()
