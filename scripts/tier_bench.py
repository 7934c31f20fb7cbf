"""Times the tiered plane kernels (K2, K3b, const) at config 3 with the real peak
states, with every state forced peaked, and with every state forced mixed."""
import ctypes
import sys
import os
import numpy as np
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import fcdiff_b200 as fcdiff
from fcdiff_b200 import _dev, _lib

(N, H, U) = (int(sys.argv[1]) if len(sys.argv) > 1 else 400, 500, 500)
iters = int(sys.argv[2]) if len(sys.argv) > 2 else 3
lib = _lib.load()
C = N * (N - 1) // 2
m = fcdiff.UnsharedRegionModel()
(_, _, _, _, b, bt) = m.sample_device(N, H, U)
fit = fcdiff.fit.UnsharedRegionFit()
fit.model = fcdiff.UnsharedRegionModel()
fit.model.eta += 0.1
fit.b, fit.bt = b, bt
fit.max_iters = iters
fit.rel_tol = -1
fit.run()
inp = fit._ensure_cache()
(lqF, qF) = fit._mF.get_dev()
(lqR, qR) = fit._mR.get_dev()
(fstate, rstate) = (fit._mF.get_state(), fit._mR.get_state())
print("peaked q_F %.4f  peaked q_R %.4f" % (float((fstate < 3).float().mean()), float((rstate < 2).float().mean())))
th = fit._theta()
ws = _dev.workspace()
(P, pitch, pitchS) = (inp['P'], inp['pitchU'], rstate.shape[1])
out = _dev.empty((4,))
lq = _dev.empty((C * 3,))


def timeit(fn, reps=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / reps


def variants():
    r_peak = rstate.clone()
    r_peak[r_peak == 2] = 0
    r_mixed = rstate.clone()
    r_mixed[r_mixed < 2] = 2
    f_mixed = torch.full_like(fstate, 3)
    return [("real", fstate, rstate), ("all peaked", fstate, r_peak), ("R mixed", fstate, r_mixed),
            ("F+R mixed", f_mixed, r_mixed)]


PROFILE = os.environ.get("FCD_PROFILE") == "1"
for (name, fst, rst) in variants():
    def elm(grad=1):
        _lib.check(lib.fcd_elm_obj_grad(_dev.ptr(P), C * pitch, C, U, pitch, _dev.ptr(qF), _dev.ptr(fst), _dev.ptr(qR),
                                        _dev.ptr(rst), pitchS, N, _dev.ptr(inp['nm']), ctypes.byref(th), grad,
                                        _dev.ptr(out), _dev.ptr(ws), _dev.stream()))

    def const():
        _lib.check(lib.fcd_elm_const(_dev.ptr(inp['L']), C, U, pitch, _dev.ptr(qF), _dev.ptr(fst), _dev.ptr(qR),
                                     _dev.ptr(rst), pitchS, N, _dev.ptr(inp['nm']), _dev.ptr(out[3:]), _dev.ptr(ws),
                                     _dev.stream()))

    def k2():
        _lib.check(lib.fcd_estep_qF(_dev.ptr(inp['S1']), _dev.ptr(inp['S2']), None, H, _dev.ptr(P), C * pitch, C, U, pitch,
                                    _dev.ptr(qR), _dev.ptr(rst), pitchS, N, _dev.ptr(inp['nm']), ctypes.byref(th),
                                    _dev.ptr(lq), None, _dev.stream()))
    if PROFILE:
        if name in ("real", "all peaked"):
            for f in (elm, const, k2):
                f()
            torch.cuda.synchronize()
            torch.cuda.cudart().cudaProfilerStart()
            for f in (elm, const, k2):
                f()
            torch.cuda.synchronize()
            torch.cuda.cudart().cudaProfilerStop()
        continue
    gb = 8e-9 * C * U
    (t1, t0, t2, t3) = (timeit(elm), timeit(lambda: elm(0)), timeit(const), timeit(k2))
    print("%-11s K3b grad %.3f ms (%.0f GB/s)  obj-only %.3f ms  const %.3f ms (%.0f GB/s)  K2 %.3f ms (%.0f GB/s alg)"
          % (name, t1, gb / t1 * 1e3, t0, t2, gb / t2 * 1e3, t3, gb / t3 * 1e3))
