#!/usr/bin/env python
"""
connections_bench.py -- posteriors of anomalous connections and patient connection states
(UnsharedRegionFit.connection_posteriors).

    python scripts/connections_bench.py [--repeat 5]

Workload: BASELINE.json configs[2] (Schaefer-400, 79,800 edges; 500 controls + 500 patients) fitted on one GPU
for the usual 10 iterations from theta_true with eta + 0.1; ONE model draw of 500 + 1000 subjects, the last 500
held out.  Read-outs: (a) the fitted cohort with maps=True and maps=False; (b) the 500 held-out patients after
score_patients, maps=True and maps=False.  Prints one JSON line:
  per point: the device times of the rows and finish kernels (torch.profiler, in a pass of its own) and the
  CUDA-event time of the whole C-ABI call; the end-to-end host time of the call (median, it returns host
  arrays); the kernel's algorithmic bytes -- planes 8 B per element on peaked edges without maps, 24 B with
  maps or on unpeaked edges; 16 B of q_R per element; writes 8 B q_T (scratch without maps) + 24 B q_F~ --
  over the rows + finish time, as a fraction of the device-to-device copy rate measured in the same run; with
  maps, the AUC of q_T against the sampler's t and the accuracy of argmax q_F~ against its f~;
  the GPU's name and power limit, read in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from patients_bench import copy_rate, gpu_name_and_power      # noqa: E402  (scripts/ is on sys.path)


def auc(torch, score, label):
    """Area under the ROC curve of a score against boolean labels (midranks for ties), on the GPU."""
    s = torch.as_tensor(score).cuda().reshape(-1)
    y = torch.as_tensor(label).cuda().reshape(-1).bool()
    (ss, idx) = torch.sort(s)
    (_, inv, counts) = torch.unique_consecutive(ss, return_inverse=True, return_counts=True)
    ends = torch.cumsum(counts, 0).double()
    mid = ends - (counts.double() - 1.0) / 2.0
    ys = y[idx]
    n1 = float(ys.sum())
    n0 = float(ys.numel()) - n1
    return (float(mid[inv][ys].sum()) - n1 * (n1 + 1) / 2.0) / (n1 * n0)


def kernel_ms(torch, call):
    """Device time per launch (ms) of the rows and finish kernels over one profiled call."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        for (tag, name) in (("rows", "connection_rows_kernel"), ("finish", "connection_finish_kernel")):
            if name in ev.key:
                total = getattr(ev, "device_time_total", None)
                if total is None:
                    total = ev.cuda_time_total
                out[tag] = out.get(tag, 0.0) + total / 1e3 / max(ev.count, 1)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeat", type=int, default=5, help="end-to-end calls per point (median reported)")
    args = ap.parse_args()

    import torch
    import fcdiff_b200 as fcdiff
    from fcdiff_b200 import _dev

    torch.cuda.set_device(0)
    (N, H, U, Uh) = (400, 500, 500, 500)
    C = N * (N - 1) // 2
    truth_model = fcdiff.UnsharedRegionModel()
    (_, t, _, ft, b, bt) = truth_model.sample_device(N, H, U + Uh)
    fit = fcdiff.fit.UnsharedRegionFit()
    (fit.b, fit.bt) = (b, bt[:, :U].contiguous())
    fit.model = fcdiff.UnsharedRegionModel()
    fit.model.eta += 0.1
    fit.max_iters = 10
    fit.rel_tol = -1.0
    fit.run()
    fstate = fit._mF.get_state()[:C].cpu().numpy()
    peaked = int((fstate < 3).sum())
    held = bt[:, U:].contiguous()
    s = fit.score_patients(held)
    peak_bw = copy_rate(torch)
    ft_state = (ft[..., 1] + 2 * ft[..., 2]).long()              # (C, U + Uh) sampled state of every connection

    out = dict(workload="connection_posteriors after a 10-iteration fit, N=%d, %d controls + %d patients; "
                        "%d held-out patients" % (N, H, U, Uh),
               gpu=gpu_name_and_power(), copy_peak_bytes_per_s=peak_bw, peaked_edges=peaked, edges=C,
               held_out_sweeps=s.sweeps, points=[])
    for (name, cols, call_args) in (("cohort", slice(0, U), ()), ("held_out", slice(U, U + Uh), (held, s.lq_R))):
        P = cols.stop - cols.start
        for maps in (True, False):
            call = lambda: fit.connection_posteriors(*call_args, maps=maps)
            r = call()                                            # warm-up: module loads, allocator
            times = []
            for _ in range(args.repeat):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                r = call()
                times.append(time.perf_counter() - t0)
            fit.profile = _dev.KernelTimers()
            call()
            call_ms = fit.profile.launch_ms("P3_connection_posteriors")[0]
            fit.profile = None
            kms = kernel_ms(torch, call)
            planes = (24 * C if maps else 8 * peaked + 24 * (C - peaked)) * P
            kbytes = planes + 16 * C * P + (8 + (24 if maps else 0)) * C * P
            kernel_s = (kms.get("rows", float("nan")) + kms.get("finish", 0.0)) * 1e-3
            pt = dict(point=name, patients=P, maps=maps, e2e_ms=1e3 * float(np.median(times)),
                      e2e_ms_all=[1e3 * x for x in times], call_event_ms=call_ms, kernel_ms=kms,
                      kernel_algorithmic_bytes=kbytes, kernel_bytes_per_s=kbytes / kernel_s,
                      kernel_fraction_of_copy_peak=kbytes / kernel_s / peak_bw,
                      expected_anomalous_mean=float(np.mean(r.expected_anomalous)),
                      true_anomalous_mean=float(t[:, cols].double().sum(0).mean()))
            if maps:
                pt["auc_q_T_vs_t"] = auc(torch, r.q_T, t[:, cols])
                pred = torch.from_numpy(r.q_F_tilde).cuda().argmax(dim=-1)
                pt["argmax_q_F_tilde_accuracy"] = float((pred == ft_state[:, cols]).double().mean())
            del r
            out["points"].append(pt)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
