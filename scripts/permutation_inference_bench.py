#!/usr/bin/env python
"""
permutation_inference_bench.py -- cost of the permutation inference (sweep.permutation_inference) over the plain
permutation sweep, and of the max-T counting kernel (fcd_maxt_counts).

    python scripts/permutation_inference_bench.py [--permutations 63] [--repeat 3] [--launches 20]

Workload: BASELINE.json configs[4]'s shape on one GPU -- Schaefer-400 (79,800 edges) x 500 controls + 500
patients from the device sampler, every fit from the reference's defaults with eta + 0.1 (bench.run_cfg5).
permutation_sweep and permutation_inference run on the same permutations, ``--repeat`` times each, alternating,
after one warm-up call of each.  Prints one JSON line:
  ms per replica of each (host clock around calls that end in a device synchronise) and the overhead of the
  inference, and the parts of one replica's row (the connection launch's device time from CUDA events over
  10 calls, and the host time of the region row's exp and mean); the device time of fcd_maxt_counts for the
  region family (400 columns) and the connection family (79,800 columns) at R1 = 1001, K = 80,200 (CUDA
  events around ``--launches`` launches after warm-up; the
  1001 x 80,200 matrix is 642 MB, beyond L2), with the bytes the three passes move (computed from the shapes
  below) and the rate they imply; the end-to-end time of sweep.maxt_pvalues at that size (host sort and
  downloads included); the GPU's name and power limit, read in the same run.
"""
import argparse
import copy
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from patients_bench import gpu_name_and_power      # noqa: E402  (scripts/ is on sys.path)


def maxt_bytes(R1, Kf):
    """Bytes of one fcd_maxt_counts call on a family of Kf columns: the gather reads the R1 x Kf values and
    the order once and writes the sorted copy; the chunk maxima (R1 x Kf / 512) are written, read and written
    again by the carry pass and read by the count pass; the count pass reads the sorted copy; 2 x 8 Kf bytes of
    counts are zeroed and added to."""
    chunks = -(-Kf // 512)
    return 8 * R1 * Kf * 3 + 8 * Kf + 8 * R1 * chunks * 4 + 8 * Kf * 4


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--permutations", type=int, default=63)
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--launches", type=int, default=20)
    args = ap.parse_args()

    import torch
    import fcdiff_b200 as fcdiff
    from fcdiff_b200 import _dev, _lib, sweep

    torch.cuda.set_device(0)
    (N, H, U) = (400, 500, 500)
    C = N * (N - 1) // 2
    model = fcdiff.UnsharedRegionModel()
    (_, _, _, _, b, bt) = model.sample_device(N, H, U)
    corr = torch.cat([b, bt], dim=1)
    labels = np.r_[np.zeros(H, bool), np.ones(U, bool)]
    start = fcdiff.UnsharedRegionModel()
    start.eta += 0.1
    streams = sweep.default_streams(1)
    R = args.permutations + 1

    def run_sweep():
        return sweep.permutation_sweep(corr, labels, args.permutations, model=start, streams=streams)

    def run_inference():
        return sweep.permutation_inference(corr, labels, args.permutations, model=start, streams=streams)

    def timed(call):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = call()
        torch.cuda.synchronize()
        return time.perf_counter() - t0, r

    timed(run_sweep)                                             # warm-up: every stream's buffers and modules
    timed(run_inference)
    (t_sweep, t_inf) = ([], [])
    for _ in range(args.repeat):
        t_sweep.append(timed(run_sweep)[0])
        (dt, res) = timed(run_inference)
        t_inf.append(dt)
    iters = int(sum(r["iterations"] for r in res.replicas.values()))
    del res

    # one replica's row at this shape: the connection launch (CUDA events) and the host part of the region row
    fit = fcdiff.fit.UnsharedRegionFit()
    fit.model = copy.deepcopy(start)
    (fit.b, fit.bt) = (b, bt)
    fit.run()
    row = _dev.empty((C,))
    fit._connection_rate_into(row)
    (s, e) = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    s.record()
    for _ in range(10):
        fit._connection_rate_into(row)
    e.record()
    e.synchronize()
    conn_ms = s.elapsed_time(e) / 10
    t0 = time.perf_counter()
    for _ in range(10):
        q1 = np.exp(fit._lq_R[:, :, 1])
        q1.mean(axis=1)
    region_host_ms = 1e3 * (time.perf_counter() - t0) / 10
    del fit, row

    # fcd_maxt_counts at R1 = 1001, K = 80,200 (two families), device time from CUDA events
    lib = _lib.load()
    (R1, K) = (1001, N + C)
    T = torch.randn((R1, K), dtype=torch.float64, device="cuda")
    obs = T[0].cpu().numpy()
    fams = {"regions": (0, N), "connections": (N, K)}
    ws = _dev.empty((int(lib.fcd_maxt_ws_bytes(R1, C)) // 8,))
    kernel = {}
    for (name, (a, b_)) in fams.items():
        order = _dev.upload(np.lexsort((np.arange(b_ - a), obs[a:b_])) + a, np.int64)
        (cu, cs) = (_dev.empty((b_ - a,), torch.int64), _dev.empty((b_ - a,), torch.int64))

        def launch():
            _lib.check(lib.fcd_maxt_counts(_dev.ptr(T), R1, K, K, _dev.ptr(order), a, b_, _dev.ptr(cu), _dev.ptr(cs),
                                           _dev.ptr(ws), _dev.stream()), "fcd_maxt_counts")
        for _ in range(3):
            launch()
        (s, e) = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        s.record()
        for _ in range(args.launches):
            launch()
        e.record()
        e.synchronize()
        ms = s.elapsed_time(e) / args.launches
        nbytes = maxt_bytes(R1, b_ - a)
        kernel[name] = dict(columns=b_ - a, ms=ms, bytes=nbytes, bytes_per_s=nbytes / (ms * 1e-3))
    fams_list = list(fams.values())
    sweep.maxt_pvalues(T, fams_list)
    e2e = []
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sweep.maxt_pvalues(T, fams_list)
        e2e.append(time.perf_counter() - t0)

    (ms_sweep, ms_inf) = (1e3 * np.median(t_sweep) / R, 1e3 * np.median(t_inf) / R)
    out = dict(workload="Schaefer-400 (79,800 edges) x 500 + 500 subjects, %d permutations + the observed "
                        "labelling, one GPU, %d replicas in flight" % (args.permutations, streams),
               gpu=gpu_name_and_power(), replicas=R, em_iterations_per_inference=iters,
               sweep_ms_per_replica=ms_sweep, inference_ms_per_replica=ms_inf,
               overhead=ms_inf / ms_sweep - 1.0,
               row_parts=dict(connection_launch_ms=conn_ms, connection_launch_share_of_sweep=conn_ms / ms_sweep,
                              region_row_host_ms=region_host_ms),
               sweep_seconds_all=t_sweep, inference_seconds_all=t_inf,
               maxt_counts=dict(R1=R1, K=K, launches=args.launches, families=kernel,
                                both_families_ms=sum(v["ms"] for v in kernel.values())),
               maxt_pvalues_e2e_ms=1e3 * float(np.median(e2e)))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
