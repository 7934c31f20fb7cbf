#!/usr/bin/env python
"""
missing_bench.py -- fits and read-outs with missing entries marginalised (UnsharedRegionFit.missing).

    python scripts/missing_bench.py [--repeat 3]

Workload: BASELINE.json configs[2] (Schaefer-400, 79,800 edges, 500 controls + 500 patients), one model draw on the
device, 10 iterations from theta_true with eta + 0.1.  Prints one JSON line:
  the time of fit.run() (host clock around a call that ends in a synchronise; median of --repeat, alternated) for
    the default path, the masked path on the same complete data, and the masked path with 10 % of the
    (region, subject) pairs dropped out (every edge of a dropped region NaN in that subject);
  fcd_resp_cache and fcd_healthy_stats alone in their missing-entry forms (missing=1: the flag, or an S0 output;
    CUDA events around 20 launches on the dropout data): their algorithmic bytes over their time, as a fraction of
    the device-to-device copy rate measured in the same run, beside their complete-data forms (missing=0) on the
    complete data;
  classify_subjects end to end on 500 + 500 held-out columns of the same draw with the same dropout;
  the GPU's name and power limit, read in the same run.
"""
import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from subjects_bench import copy_rate, gpu_name_and_power    # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeat", type=int, default=3, help="fits per path (median reported)")
    args = ap.parse_args()

    import torch
    import fcdiff_b200 as fcdiff
    from fcdiff_b200 import _dev, _lib

    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    (N, H, U) = (400, 500, 500)
    C = N * (N - 1) // 2
    (_, _, _, _, b, bt) = fcdiff.UnsharedRegionModel().sample_device(N, 2 * H, 2 * U)
    n = torch.as_tensor(np.repeat(np.arange(N), np.arange(N)), device=dev)          # edge c = n (n - 1) / 2 + m
    m = torch.as_tensor(np.concatenate([np.arange(i) for i in range(N)]), device=dev)

    def dropout(x, seed):
        g = torch.Generator(device=dev).manual_seed(seed)
        drop = torch.rand((N, x.shape[1]), generator=g, device=dev) < 0.10
        return torch.where(drop[n] | drop[m], torch.full_like(x, float("nan")), x)

    data = dict(complete=(b[:, :H].contiguous(), bt[:, :U].contiguous()))
    data["dropout"] = (dropout(data["complete"][0], 1), dropout(data["complete"][1], 2))

    def run(missing, which):
        fit = fcdiff.fit.UnsharedRegionFit()
        (fit.b, fit.bt) = data[which]
        fit.model = fcdiff.UnsharedRegionModel()
        fit.model.eta += 0.1
        fit.max_iters = 10
        fit.rel_tol = -1.0
        fit.missing = missing
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fit.run()
        torch.cuda.synchronize()
        return time.perf_counter() - t0, fit

    paths = (("default", "reject", "complete"), ("masked_complete", "marginalize", "complete"),
             ("masked_dropout", "marginalize", "dropout"))
    for (_, missing, which) in paths:                                 # warm-up: modules, allocator, tables
        run(missing, which)
    times = {name: [] for (name, _, _) in paths}
    fits = {}
    for _ in range(args.repeat):
        for (name, missing, which) in paths:
            (t, fits[name]) = run(missing, which)
            times[name].append(t)
    peak_bw = copy_rate(torch)

    # the two masked set-up kernels alone, against their unmasked forms on the complete data
    lib = _lib.load()
    fit = fits["masked_dropout"]
    th = fit._theta()
    P = _dev.empty((4, C, U))
    (S1, S2, S0) = (_dev.empty((C,)), _dev.empty((C,)), _dev.empty((C,)))
    (bd, btd) = data["dropout"]
    (bc, btc) = data["complete"]
    calls = {
        "resp_cache missing=1": lambda: lib.fcd_resp_cache(_dev.ptr(btd), C, U, U, ctypes.byref(th), _dev.ptr(P),
                                                           C * U, _dev.ptr(P[3]), 1, _dev.stream()),
        "resp_cache missing=0": lambda: lib.fcd_resp_cache(_dev.ptr(btc), C, U, U, ctypes.byref(th), _dev.ptr(P),
                                                           C * U, _dev.ptr(P[3]), 0, _dev.stream()),
        "healthy_stats missing=1": lambda: lib.fcd_healthy_stats(_dev.ptr(bd), C, H, H, _dev.ptr(S1), _dev.ptr(S2),
                                                                 _dev.ptr(S0), _dev.stream()),
        "healthy_stats missing=0": lambda: lib.fcd_healthy_stats(_dev.ptr(bc), C, H, H, _dev.ptr(S1), _dev.ptr(S2),
                                                                 None, _dev.stream())}
    algo_bytes = {"resp_cache missing=1": 8 * C * U * 5, "resp_cache missing=0": 8 * C * U * 5,
                  "healthy_stats missing=1": 8 * C * H + 24 * C, "healthy_stats missing=0": 8 * C * H + 16 * C}
    kernels = {}
    for (name, call) in calls.items():
        _lib.check(call(), name)
        reps = 20
        (e0, e1) = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        e0.record()
        for _ in range(reps):
            _lib.check(call(), name)
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1) / reps
        kernels[name] = dict(ms=ms, algorithmic_bytes=algo_bytes[name],
                             fraction_of_copy_peak=algo_bytes[name] / (ms * 1e-3) / peak_bw)

    # classify_subjects on held-out columns with the same dropout
    held = dropout(torch.cat([b[:, H:], bt[:, U:]], dim=1).contiguous(), 3)
    fit.classify_subjects(held)
    ctimes = []
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        c = fit.classify_subjects(held)
        ctimes.append(time.perf_counter() - t0)
    truth = np.arange(held.shape[1]) >= H

    med = {k: 1e3 * float(np.median(v)) for (k, v) in times.items()}
    res = dict(
        workload="fit.run() 10 iterations, N=%d (%d edges), %d + %d; dropout: 10 %% of (region, subject) pairs"
                 % (N, C, H, U),
        gpu=gpu_name_and_power(), copy_peak_bytes_per_s=peak_bw,
        fit_ms=med, fit_ms_all={k: [1e3 * t for t in v] for (k, v) in times.items()},
        masked_over_default=med["masked_complete"] / med["default"],
        dropout_over_default=med["masked_dropout"] / med["default"],
        bit_identical_without_nan=bool(fits["default"].energy == fits["masked_complete"].energy),
        missing_fraction_patients=float(torch.isnan(data["dropout"][1]).double().mean()),
        kernels=kernels,
        classify_ms=1e3 * float(np.median(ctimes)), classify_subjects=int(held.shape[1]),
        classify_accuracy=float(np.mean((c.p_patient > 0.5) == truth)))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
