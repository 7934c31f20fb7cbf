"""Where the end-to-end time of fit.run(max_iters=1) from pinned host arrays goes (config 3)."""
import os, sys, time
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import fcdiff_b200 as fcdiff
from fcdiff_b200 import _dev

(N, H, U) = (400, 500, 500)
m = fcdiff.UnsharedRegionModel()
(_, _, _, _, b, bt) = m.sample_device(N, H, U)
bh = torch.empty(b.shape, dtype=torch.float64).pin_memory(); bh.copy_(b)
bth = torch.empty(bt.shape, dtype=torch.float64).pin_memory(); bth.copy_(bt)
(bn, btn) = (bh.numpy(), bth.numpy())

def sync(): torch.cuda.synchronize(); return time.perf_counter()

for rep in range(3):
    fit = fcdiff.fit.UnsharedRegionFit(); fit.model = fcdiff.UnsharedRegionModel(); fit.model.eta += 0.1
    fit.b, fit.bt = bn, btn
    t0 = sync()
    fit._init_lps(N, H, U); t1 = sync()
    fit._ensure_inputs(); t2 = sync()
    fit._update_lps(); fit._ensure_cache(); t3 = sync()
    fit._ensure_patient_planes(); t4 = sync()
    e0 = fit._eval_energy(); t5 = sync()
    fit._update_lq_F(); t6 = sync()
    fit._update_lq_R(); t7 = sync()
    fit._update_theta(); t8 = sync()
    fit._update_lps(); e1 = fit._eval_energy(); t9 = sync()
    a = fit._lq_F; c = fit._lq_R; t10 = sync()
    if rep == 2:
        names = ["init_lps", "upload+healthy", "resp_cache", "patient_planes", "energy0", "K2", "K2b", "theta(nfev=%d)" % fit.n_objective_evals[-1] if fit.n_objective_evals else "theta", "energy1", "download"]
        ts = [t0, t1, t2, t3, t4, t5, t6, t7, t8, t9, t10]
        for i, nm in enumerate(names):
            print("%-18s %7.2f ms" % (nm, (ts[i + 1] - ts[i]) * 1e3))
        print("total %.2f ms" % ((t10 - t0) * 1e3))
# raw H2D rate
x = torch.empty(bh.shape, dtype=torch.float64, device="cuda")
for _ in range(2):
    t0 = sync(); x.copy_(bh, non_blocking=True); t1 = sync()
print("H2D %.1f MB in %.2f ms = %.1f GB/s" % (bh.numel() * 8 / 1e6, (t1 - t0) * 1e3, bh.numel() * 8 / (t1 - t0) / 1e9))
