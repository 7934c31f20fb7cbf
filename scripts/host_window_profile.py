"""Host time per step function of run() in the settled iterations of a fresh config-3 fit (perf_counter around the
calls; the GPU work is asynchronous except for the two waits inside _update_theta): what the host spends between
the solver wait and the launch of the next sweep -- the window the speculative E-step has to cover."""
import os, sys, time, collections
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import fcdiff_b200 as fcdiff

(N, H, U) = (400, 500, 500)
(_, _, _, _, b, bt) = fcdiff.UnsharedRegionModel().sample_device(N, H, U)
acc = collections.defaultdict(list)


def wrap(fit, name):
    f = getattr(fit, name)

    def g(*a, **k):
        t0 = time.perf_counter()
        r = f(*a, **k)
        acc[name].append((time.perf_counter() - t0) * 1e6)
        return r
    setattr(fit, name, g)


for rep in range(3):
    fit = fcdiff.fit.UnsharedRegionFit(); fit.model = fcdiff.UnsharedRegionModel(); fit.model.eta += 0.1
    (fit.b, fit.bt) = (b, bt); fit.max_iters = 10; fit.rel_tol = -1.0
    if rep == 2:
        for n in ("_update_lq_F", "_update_lq_R", "_update_theta", "_update_lps", "_eval_energy", "_is_converged",
                  "_ensure_inputs", "_ensure_cache", "_ensure_patient_planes", "_theta", "_energy_key", "_speculative_estep",
                  "_update_pi_gamma", "_update_theta_sub", "_solver_context", "_build_streams"):
            wrap(fit, n)
    torch.cuda.synchronize(); t0 = time.perf_counter(); fit.run(); torch.cuda.synchronize()
    print("fit %d: %.3f ms" % (rep, (time.perf_counter() - t0) * 1e3))
for (k, v) in acc.items():
    v2 = v[len(v) // 2:]
    print("%-24s calls %3d  median %7.1f us  (second half of the fit: median %7.1f us, sum/iter %7.1f us)" % (
        k, len(v), float(np.median(v)), float(np.median(v2)), float(np.sum(v2)) / 5.0))
