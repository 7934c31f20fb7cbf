#!/usr/bin/env python
"""
patients_bench.py -- scoring held-out patients with a fitted model (UnsharedRegionFit.score_patients).

    python scripts/patients_bench.py [--patients 500,1] [--repeat 5]

Workload: BASELINE.json configs[2] (Schaefer-400, 79,800 edges; 500 controls + 500 patients) fitted on one GPU
for the usual 10 iterations from theta_true with eta + 0.1, then held-out patients drawn from the same model --
ONE model draw of 500 + max(--patients) patients, split into columns -- are scored from device-resident
correlations with the default max_sweeps / tol.  Prints one JSON line:
  per point (number of scored patients): CUDA-event times of every stage (planes, region weights, each sweep,
  each change reduction, the per-patient terms), the sweep count, end-to-end time and patients per second
  (host clock around score_patients, which returns host arrays), the terms kernel's algorithmic bytes
  (16 B per edge-patient on peaked edges, 32 B on unpeaked ones, plus 16 N U' of q_R) over its time as a
  fraction of the device-to-device copy rate measured in the same run, and MAP recall / precision of the
  planted anomalous regions;
  the GPU's name and power limit, read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def gpu_name_and_power():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def copy_rate(torch):
    """Device-to-device copy rate (bytes read + written per second) of a 2 GB buffer."""
    x = torch.empty(1 << 28, dtype=torch.float64, device="cuda")
    y = torch.empty_like(x)
    y.copy_(x)
    (s, e) = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    reps = 10
    s.record()
    for _ in range(reps):
        y.copy_(x)
    e.record()
    e.synchronize()
    return 2.0 * x.numel() * 8 * reps / (s.elapsed_time(e) * 1e-3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--patients", default="500,1", help="comma-separated numbers of held-out patients to score")
    ap.add_argument("--repeat", type=int, default=5, help="end-to-end calls per point (median reported)")
    args = ap.parse_args()
    points = [int(p) for p in args.patients.split(",")]

    import torch
    import fcdiff_b200 as fcdiff
    from fcdiff_b200 import _dev

    torch.cuda.set_device(0)
    (N, H, U) = (400, 500, 500)
    C = N * (N - 1) // 2
    truth_model = fcdiff.UnsharedRegionModel()
    (r, _, _, _, b, bt) = truth_model.sample_device(N, H, U + max(points))
    r = r.cpu().numpy() > 0
    fit = fcdiff.fit.UnsharedRegionFit()
    (fit.b, fit.bt) = (b, bt[:, :U].contiguous())
    fit.model = fcdiff.UnsharedRegionModel()
    fit.model.eta += 0.1
    fit.max_iters = 10
    fit.rel_tol = -1.0
    fit.run()
    fstate = fit._mF.get_state()[:C].cpu().numpy()
    peaked = int((fstate < 3).sum())
    peak_bw = copy_rate(torch)

    out = dict(workload="score_patients after a 10-iteration fit, N=%d, %d controls + %d patients" % (N, H, U),
               gpu=gpu_name_and_power(), copy_peak_bytes_per_s=peak_bw, peaked_edges=peaked, edges=C,
               fit_energy=fit.energy[-1], points=[])
    for P in points:
        held = bt[:, U:U + P].contiguous()
        fit.score_patients(held)                                  # warm-up: module loads, allocator, log table
        times = []
        for _ in range(args.repeat):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            s = fit.score_patients(held)
            times.append(time.perf_counter() - t0)
        e2e = float(np.median(times))
        fit.profile = _dev.KernelTimers()
        s = fit.score_patients(held)
        stages = {name: fit.profile.launch_ms(name) for name in
                  ("P0_resp_cache", "K2b_region_weights", "K2b_sweep", "P1_qR_change", "P2_patient_terms")}
        fit.profile = None
        terms_ms = stages["P2_patient_terms"][0]
        terms_bytes = 16 * peaked * P + 32 * (C - peaked) * P + 16 * N * P
        pred = s.lq_R[:, :, 1] > s.lq_R[:, :, 0]
        truth = r[:, U:U + P]
        tp = float((pred & truth).sum())
        out["points"].append(dict(
            patients=P, sweeps=s.sweeps, max_change=s.max_change, e2e_ms=1e3 * e2e,
            e2e_ms_all=[1e3 * t for t in times], patients_per_s=P / e2e,
            stage_ms=dict(planes=stages["P0_resp_cache"], weights=stages["K2b_region_weights"],
                          sweeps=stages["K2b_sweep"], change=stages["P1_qR_change"], terms=stages["P2_patient_terms"]),
            terms_algorithmic_bytes=terms_bytes, terms_bytes_per_s=terms_bytes / (terms_ms * 1e-3),
            terms_fraction_of_copy_peak=terms_bytes / (terms_ms * 1e-3) / peak_bw,
            recall=tp / max(float(truth.sum()), 1.0), precision=tp / max(float(pred.sum()), 1.0),
            anomaly_score_mean=float(np.mean(s.free_energy_typical - s.free_energy))))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
