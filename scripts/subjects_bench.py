#!/usr/bin/env python
"""
subjects_bench.py -- classifying held-out subjects of unknown group with a fitted model
(UnsharedRegionFit.classify_subjects) and cross-validating it (sweep.cross_validate).

    python scripts/subjects_bench.py [--repeat 5] [--folds 5]

Workload: BASELINE.json configs[2] (Schaefer-400, 79,800 edges).  ONE model draw of 1000 controls + 1000 patients;
the first 500 + 500 are fitted on one GPU for the usual 10 iterations from theta_true with eta + 0.1, the other
500 + 500 are classified from device-resident correlations with the default prior (the fit's 500 / 1000), max_sweeps
and tol.  Prints one JSON line:
  the end-to-end time of classify_subjects (host clock around a call that returns host arrays, median of --repeat);
  CUDA-event times of every stage (planes, region weights, each sweep, each change reduction, the per-patient terms,
  the control terms);
  fcd_control_terms alone (CUDA events around 20 launches on the held-out columns): its algorithmic bytes
  8 C S + 24 C over its time, as a fraction of the device-to-device copy rate measured in the same run;
  AUC and accuracy (p_patient > 1/2) of the held-out subjects;
  the time of a --folds-fold cross_validate of the fitted cohort (500 + 500, 10 iterations per fold);
  the GPU's name and power limit, read in the same run.
"""
import argparse
import ctypes
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


def auc(pos, neg):
    """Mann-Whitney AUC: the probability that a positive outscores a negative (ties count half)."""
    import scipy.stats
    ranks = scipy.stats.rankdata(np.concatenate([pos, neg]))
    return float((ranks[:len(pos)].sum() - len(pos) * (len(pos) + 1) / 2.0) / (len(pos) * len(neg)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeat", type=int, default=5, help="end-to-end calls (median reported)")
    ap.add_argument("--folds", type=int, default=5, help="folds of the cross-validation")
    args = ap.parse_args()

    import torch
    import fcdiff_b200 as fcdiff
    from fcdiff_b200 import _dev, _lib, sweep

    torch.cuda.set_device(0)
    (N, H, U) = (400, 500, 500)
    C = N * (N - 1) // 2
    truth_model = fcdiff.UnsharedRegionModel()
    (_, _, _, _, b, bt) = truth_model.sample_device(N, 2 * H, 2 * U)
    fit = fcdiff.fit.UnsharedRegionFit()
    (fit.b, fit.bt) = (b[:, :H].contiguous(), bt[:, :U].contiguous())
    fit.model = fcdiff.UnsharedRegionModel()
    fit.model.eta += 0.1
    fit.max_iters = 10
    fit.rel_tol = -1.0
    fit.run()
    peak_bw = copy_rate(torch)

    held = torch.cat([b[:, H:], bt[:, U:]], dim=1).contiguous()       # 500 controls, then 500 patients
    S = int(held.shape[1])
    truth = np.arange(S) >= H
    fit.classify_subjects(held)                                        # warm-up: module loads, allocator, log table
    times = []
    for _ in range(args.repeat):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        c = fit.classify_subjects(held)
        times.append(time.perf_counter() - t0)
    fit.profile = _dev.KernelTimers()
    c = fit.classify_subjects(held)
    names = ("P0_resp_cache", "K2b_region_weights", "K2b_sweep", "P1_qR_change", "P2_patient_terms",
             "P4_control_terms")
    stages = {name: fit.profile.launch_ms(name) for name in names}
    fit.profile = None

    # fcd_control_terms alone, on the held-out columns (S even: no padding)
    lib = _lib.load()
    th = fit._theta(use_snapshot=False)
    qF = fit._mF.get_dev()[1]
    out = _dev.empty((S,))
    ws = _dev.empty((int(lib.fcd_control_terms_ws_bytes(C, S)) // 8,))
    call = lambda: _lib.check(lib.fcd_control_terms(_dev.ptr(held), C, S, S, _dev.ptr(qF), ctypes.byref(th),
                                                    _dev.ptr(out), _dev.ptr(ws), 0, _dev.stream()), "fcd_control_terms")
    call()
    reps = 20
    (e0, e1) = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    e0.record()
    for _ in range(reps):
        call()
    e1.record()
    e1.synchronize()
    control_ms = e0.elapsed_time(e1) / reps
    control_bytes = 8 * C * S + 24 * C

    # cross-validation of the fitted cohort
    corr = torch.cat([b[:, :H], bt[:, :U]], dim=1).contiguous()
    labels = np.arange(H + U) >= H
    opts = dict(max_iters=10, rel_tol=-1.0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    cv = sweep.cross_validate(corr, labels, n_folds=args.folds, fit_options=opts)
    torch.cuda.synchronize()
    cv_s = time.perf_counter() - t0

    res = dict(
        workload="classify_subjects after a 10-iteration fit, N=%d, fitted on %d + %d, classifying %d + %d"
                 % (N, H, U, H, U),
        gpu=gpu_name_and_power(), copy_peak_bytes_per_s=peak_bw, edges=C, fit_energy=fit.energy[-1],
        subjects=S, sweeps=c.sweeps, max_change=c.max_change,
        e2e_ms=1e3 * float(np.median(times)), e2e_ms_all=[1e3 * t for t in times],
        stage_ms=dict(planes=stages["P0_resp_cache"], weights=stages["K2b_region_weights"],
                      sweeps=stages["K2b_sweep"], change=stages["P1_qR_change"], patient_terms=stages["P2_patient_terms"],
                      control_terms=stages["P4_control_terms"]),
        control_terms_ms=control_ms, control_terms_algorithmic_bytes=control_bytes,
        control_terms_bytes_per_s=control_bytes / (control_ms * 1e-3),
        control_terms_fraction_of_copy_peak=control_bytes / (control_ms * 1e-3) / peak_bw,
        auc=auc(c.log_odds[truth], c.log_odds[~truth]),
        accuracy=float(np.mean((c.p_patient > 0.5) == truth)),
        cv_folds=args.folds, cv_s=cv_s, cv_auc=auc(cv["log_odds"][labels], cv["log_odds"][~labels]),
        cv_accuracy=float(np.mean((cv["p_patient"] > 0.5) == labels)))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
