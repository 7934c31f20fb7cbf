#!/usr/bin/env python
"""
Cleaned correlation stage (fcd_corr_fisherz_clean) on bench.py's K1 workload: 1000 subjects x Schaefer-400 x
1200 frames of planted-factor series, generated on the device from a seed.

Variants: plain (fcd_corr_fisherz); mask only (10 % of frames censored, lengths 900 - 1200); K = 6, 24 and 36
confounds with that mask.  Per variant: the call's time from CUDA events after warm-up, and a per-kernel
split from torch.profiler in a separate pass -- basis (confound_basis_kernel), cleaning (standardise_kernel /
clean_kernel), Gram + epilogue (gram_tc_kernel) -- with algorithmic bytes and fp64 FMAs from the shapes and
their fractions of the copy rate (a 2 GiB device-to-device copy) and the fp64 rate (a 8192^3 float64
matmul) measured in the same run.  Checks that the mask variant with no frame censored has the bits of
the plain output.  Prints one JSON line.

    python scripts/clean_corr_bench.py [--subjects 1000] [--reps 5] [--seed 1]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from fcdiff_b200 import corr          # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    limit = None
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        if q.returncode == 0:
            limit = q.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pass
    return {"name": name, "nvidia_smi": limit}


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    (e0, e1) = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def rates(reps):
    n = (2 << 30) // 4
    a = torch.empty(n, dtype=torch.float32, device="cuda").fill_(1.0)
    b = torch.empty_like(a)
    ms = timed(lambda: b.copy_(a), reps)
    copy_gbs = 2 * a.numel() * 4 / (ms * 1e-3) / 1e9
    del a, b
    m = 8192
    x = torch.randn((m, m), dtype=torch.float64, device="cuda")
    y = torch.randn((m, m), dtype=torch.float64, device="cuda")
    ms = timed(lambda: torch.matmul(x, y), max(2, reps // 2))
    fp64_tflops = 2.0 * m ** 3 / (ms * 1e-3) / 1e12
    return copy_gbs, fp64_tflops


def workload(S, N, T, seed):
    """bench.py's K1 series: eight latent signals, loadings +0.55 / -0.27, 5 % sign flips among patients."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    F = 8
    U = S // 2
    fac = torch.arange(N, device="cuda") % F
    load = torch.where(torch.rand((N,), device="cuda", generator=g) < 0.5, 0.55, -0.27).to(torch.float32)
    a = load[None, :].repeat(S, 1)
    flip = torch.rand((U, N), device="cuda", generator=g) < 0.05
    a[S - U:][flip] *= -1.0
    ts = torch.randn((S, N, T), dtype=torch.float32, device="cuda", generator=g)
    ts *= torch.sqrt(1.0 - a * a)[:, :, None]
    z = torch.randn((S, F, T), dtype=torch.float32, device="cuda", generator=g)
    ts += a[:, :, None] * z[:, fac, :]
    return ts, g


def kernel_split(fn):
    """Per-kernel device time (ms) of one call, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if t <= 0:
            continue
        for (key, stage) in (("confound_basis_kernel", "basis"), ("clean_kernel", "clean"),
                             ("standardise_kernel", "clean"), ("gram_tc_kernel", "gram"),
                             ("gram_simt_kernel", "gram"), ("mark_", "mark")):
            if key in ev.key:
                out[stage] = out.get(stage, 0.0) + t / 1000.0
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--subjects", type=int, default=1000)
    ap.add_argument("--regions", type=int, default=400)
    ap.add_argument("--frames", type=int, default=1200)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=1)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("clean_corr_bench.py needs a CUDA device")
    (S, N, T) = (args.subjects, args.regions, args.frames)
    C = N * (N - 1) // 2
    Tp = (T + 31) // 32 * 32
    info = card()
    (copy_gbs, fp64_tflops) = rates(args.reps)
    (ts, g) = workload(S, N, T, args.seed)
    lengths = torch.randint(900, T + 1, (S,), device="cuda", generator=g)
    keep = (torch.rand((S, T), device="cuda", generator=g) >= 0.1) & \
        (torch.arange(T, device="cuda")[None, :] < lengths[:, None])
    n_kept = int(keep.sum())                                # kept frames, all subjects
    out = torch.empty((C, S), dtype=torch.float64, device="cuda")

    res = {"workload": "%d subjects x %d regions x %d frames (planted-factor series, seed %d)" % (S, N, T, args.seed),
           "card": info, "copy_GBps": copy_gbs, "fp64_matmul_TFLOPs": fp64_tflops, "kept_frames": n_kept,
           "variants": {}}
    plain = corr.correlations_device(ts, fisher=True).clone()
    allkept = corr.correlations_device(ts, fisher=True, sample_mask=torch.ones((S, T), dtype=torch.bool,
                                                                              device="cuda"))
    same = (plain.view(torch.int64) == allkept.view(torch.int64)) | ((plain == 0) & (allkept == 0))
    res["mask_all_kept_bit_identical"] = bool(same.all())
    del allkept
    variants = [("plain", None, 0), ("mask", keep, 0)] + [("K%d" % K, keep, K) for K in (6, 24, 36)]
    for (name, mask, K) in variants:
        conf = torch.randn((S, T, K), dtype=torch.float64, device="cuda", generator=g) if K else None

        def call():
            corr.correlations_device(ts, fisher=True, out=out, sample_mask=mask, confounds=conf)
        ms = timed(call, args.reps)
        split = kernel_split(call)
        samples = N * n_kept if mask is not None else S * N * T
        v = {"ms": ms, "stage_ms": split}
        # cleaning: 4 B read per sample (every padded frame of ts is streamed) + 8 B of Z / Zlo written per frame
        clean_bytes = S * N * (T * 4 + Tp * 8)
        v["clean_bytes"] = clean_bytes
        if "clean" in split:
            v["clean_copy_frac"] = clean_bytes / (split["clean"] * 1e-3) / 1e9 / copy_gbs
        if K:
            clean_fma = 2.0 * K * samples                      # K dot products + K axpys per kept sample
            basis_fma = 2.0 * (K * (K - 1) + 2 * K) * n_kept        # two MGS passes: dots + axpys, norms
            v.update({"clean_fp64_fma": clean_fma, "basis_fp64_fma": basis_fma,
                      "basis_bytes": S * T * K * 8 + S * K * Tp * 8})
            if "clean" in split:
                v["clean_fp64_frac"] = 2 * clean_fma / (split["clean"] * 1e-3) / 1e12 / fp64_tflops
        res["variants"][name] = v
        del conf
    print(json.dumps(res))


if __name__ == "__main__":
    main()
