"""
Replica sweeps over the fit: group-label permutations and random restarts
(BASELINE.json configs[4]; SURVEY 8e "Config 5"), and stratified k-fold
cross-validation of the two-group classifier.  The reference has neither --
it has no driver beyond ``UnsharedRegionFit.run()`` (fcdiff/fit.py:56-82) -- so
this module only orchestrates: every replica is one ordinary fit of this
package on a re-labelled (or re-initialised) copy of the problem.

Sharding: replicas, not edges.  Each rank keeps the whole (C, S) correlation
matrix and runs the replicas ``rank, rank + world, ...``; nothing is exchanged
until the results are gathered at the end (one ``all_gather_object``).
"""
import copy

import numpy as np
import torch

from . import _dev
from .fit import UnsharedRegionFit
from .model import UnsharedRegionModel


class SharedPlanes(object):
    """Responsibility planes of ALL subjects of one (C, S) correlation matrix for fixed (mu, sigma),
    built once: every relabelling of the subjects selects its controls' sufficient statistics and its
    patients' planes from them (``UnsharedRegionFit.set_shared_inputs``, csrc/fcd_replica.cu) instead of
    taking the exponentials again.

    X  [C][pitchS]       the correlations (zero padded to an even pitch)
    PL [4][C][pitchS]    p_0, p_1, p_2, L of every (edge, subject)      (fcd_resp_cache)
    nm [C]               edge table

    ``missing``: the ``UnsharedRegionFit.missing`` of the fits that use the planes; with ``"marginalize"`` a NaN
    correlation is an unobserved entry (fcd_resp_cache with missing = 1) and +-inf is rejected.
    """

    def __init__(self, corr, model, missing="reject"):
        import ctypes
        from . import _lib
        from .util import C_to_N
        lib = _lib.load()
        dev = _dev.device()
        x = corr if torch.is_tensor(corr) else torch.from_numpy(np.ascontiguousarray(corr, dtype=np.float64))
        x = x.to(dev, torch.float64)
        (C, S) = (int(x.shape[0]), int(x.shape[1]))
        if (C_to_N(C) % 1) != 0:
            raise ValueError("Number of connections (%u) must be a triangular number." % C)
        if missing not in ("reject", "marginalize"):
            raise ValueError("missing must be 'reject' or 'marginalize' (got %r)" % (missing,))
        if missing == "marginalize" and bool(torch.isinf(x).any()):
            raise ValueError("corr must hold finite correlations or NaN")
        self.missing = missing
        (self.C, self.S, self.pitchS) = (C, S, _dev.even(S))
        if self.pitchS == S:
            self.X = x.contiguous()
        else:
            self.X = _dev.zeros((C, self.pitchS))
            self.X[:, :S].copy_(x)
        th = _lib.make_theta(float(np.asarray(model.pi).reshape(-1)[-1]), model.eta, model.epsilon,
                             np.asarray(model.gamma).reshape(-1), model.mu, model.sigma)
        self.cache_key = (tuple(float(v) for v in model.mu), tuple(float(v) for v in model.sigma))
        self.PL = _dev.empty((4, C, self.pitchS))
        _lib.check(lib.fcd_resp_cache(_dev.ptr(self.X), C, S, self.pitchS, ctypes.byref(th), _dev.ptr(self.PL),
                                      C * self.pitchS, _dev.ptr(self.PL[3]), int(missing == "marginalize"),
                                      _dev.stream()), "fcd_resp_cache")
        self.nm = _dev.empty((max(C, 1),), torch.int32)
        _lib.check(lib.fcd_edge_table(0, C, _dev.ptr(self.nm), _dev.stream()), "fcd_edge_table")


def replica_indices(n_replicas, rank=0, world=1):
    """Replicas handled by ``rank``: a strided split, so that every rank gets
    the same number (+-1) whatever ``n_replicas``."""
    return list(range(rank, n_replicas, world))


def permuted_labels(labels, n_permutations, seed=0):
    """(n_permutations + 1, S) boolean array: row 0 is the observed labelling,
    row i > 0 a permutation drawn with ``RandomState(seed).permutation``
    (group sizes are preserved)."""
    labels = np.asarray(labels, dtype=bool)
    rng = np.random.RandomState(seed)
    out = np.empty((n_permutations + 1, labels.size), dtype=bool)
    out[0] = labels
    for i in range(1, n_permutations + 1):
        out[i] = labels[rng.permutation(labels.size)]
    return out


def _gather(results, group):
    import torch.distributed as dist
    if group is None and not (dist.is_available() and dist.is_initialized()):
        return results
    world = dist.get_world_size(group)
    if world == 1:
        return results
    bucket = [None] * world
    dist.all_gather_object(bucket, results, group=group)
    merged = {}
    for part in bucket:
        merged.update(part)
    return merged


def _summary(fit):
    m = fit.model
    return dict(energy=list(fit.energy), pi=float(m.pi), eta=float(m.eta), epsilon=float(m.epsilon),
                gamma=np.asarray(m.gamma, dtype=np.float64).copy(), mu=np.asarray(m.mu, dtype=np.float64).copy(),
                sigma=np.asarray(m.sigma, dtype=np.float64).copy(), iterations=len(fit.energy) - 1,
                expected_anomalous_regions=float(np.exp(fit._lq_R[:, :, 1]).sum()))


def default_streams(world=1):
    """Replicas in flight per GPU: two when the host has the cores for it (every fit in flight has one
    thread that spins on mapped memory while it waits for a result), else one."""
    import os
    return 2 if (os.cpu_count() or 1) >= 4 * max(int(world), 1) else 1


def _run_replicas(indices, run_one, streams):
    """``run_one(i) -> summary`` for every replica index, ``streams`` of them in flight on this GPU: each worker
    thread owns a CUDA stream (and, through ``_dev``, its own reduction workspace, publication window and
    solver block); while one replica's host side waits for a result, the other's kernels fill the GPU.  The
    ctypes calls and the waits release the GIL.  Results do not depend on ``streams`` (every fit is
    deterministic and self-contained)."""
    results = {}
    if streams <= 1 or len(indices) <= 1:
        for i in indices:
            results[i] = run_one(i)
        return results
    import threading
    dev = _dev.device()
    main = torch.cuda.current_stream()
    errors = []

    def worker(k, s):
        try:
            torch.cuda.set_device(dev)                   # the current device is per thread
            s.wait_stream(main)                          # the shared planes were built on the caller's stream
            with torch.cuda.stream(s):
                for i in indices[k::streams]:
                    results[i] = run_one(i)
                s.synchronize()
        except BaseException as exc:                     # re-raised by the caller
            errors.append(exc)

    ss = [torch.cuda.Stream(device=dev) for _ in range(streams)]
    threads = [threading.Thread(target=worker, args=(k, ss[k]), daemon=True) for k in range(streams)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for s in ss:
        main.wait_stream(s)
    if errors:
        raise errors[0]
    return results


def _configure(fit, options):
    for (k, v) in (options or {}).items():
        if not hasattr(fit, k):
            raise AttributeError("UnsharedRegionFit has no option %r" % k)
        setattr(fit, k, v)


def permutation_sweep(corr, labels, n_permutations, model=None, seed=0, fit_options=None, rank=0, world=1,
                      group=None, gather=True, shared_planes=True, streams=None):
    """
    Fits the model once per group labelling: the observed one and
    ``n_permutations`` random re-labellings of the subjects.

    Parameters
    ----------
    corr : (C, S) array or CUDA tensor
        Correlations of ALL subjects, one column per subject (the layout K1
        writes, ``fcdiff_b200.corr``).
    labels : (S,) bool
        True for patients (columns of ``bt``), False for controls (``b``).
    model : UnsharedRegionModel
        Initial parameters of every fit (deep-copied per replica; default: the
        reference's defaults, fcdiff/model.py:31-38).
    fit_options : dict
        Attributes set on every ``UnsharedRegionFit`` (``max_iters``, ``rel_tol``,
        ``edge_lookup``, ``missing``, ...).
    rank, world, group
        Replica sharding (see the module docstring); ``gather`` merges the
        results of all ranks.
    shared_planes : bool
        Build the responsibility planes once for all S subjects and let every
        replica select its columns from them (:class:`SharedPlanes`; default).
        With ``update_mu_sigma`` in ``fit_options`` (the planes then change during a
        fit) or ``shared_planes=False`` every replica uploads its own columns and
        rebuilds its planes -- same results.
    streams : int or None
        Replicas in flight on this GPU (one CUDA stream and one host thread each; default
        :func:`default_streams`).  Same results for any value.

    Returns
    -------
    dict replica index -> summary (energy trace, fitted parameters, expected
    number of anomalous regions); index 0 is the observed labelling.
    """
    lab = permuted_labels(labels, n_permutations, seed)
    dev = _dev.device()
    corr_dev = corr if torch.is_tensor(corr) else torch.from_numpy(np.ascontiguousarray(corr, dtype=np.float64))
    corr_dev = corr_dev.to(dev, torch.float64)
    model = UnsharedRegionModel() if model is None else model
    shared = None
    if shared_planes and not (fit_options or {}).get("update_mu_sigma"):
        shared = SharedPlanes(corr_dev, model, missing=(fit_options or {}).get("missing", "reject"))
    def run_one(i):
        pat = torch.from_numpy(np.flatnonzero(lab[i])).to(dev)
        con = torch.from_numpy(np.flatnonzero(~lab[i])).to(dev)
        fit = UnsharedRegionFit()
        fit.model = copy.deepcopy(model)
        _configure(fit, fit_options)
        if shared is not None:
            fit.set_shared_inputs(shared, con, pat)
        else:
            fit.b = corr_dev.index_select(1, con)          # column gather: data movement only
            fit.bt = corr_dev.index_select(1, pat)
        fit.run()
        return _summary(fit)

    results = _run_replicas(replica_indices(n_permutations + 1, rank, world), run_one,
                            default_streams(world) if streams is None else int(streams))
    return _gather(results, group) if gather else results


def stratified_folds(labels, n_folds=5, seed=0):
    """(S,) int array: the cross-validation fold of every subject.  Each class is shuffled with
    ``RandomState(seed)`` and dealt round robin over the folds, the patients continuing where the controls
    stopped: every fold gets each class's count over ``n_folds`` rounded down or up, and the fold sizes differ
    by at most one."""
    labels = np.asarray(labels, dtype=bool).reshape(-1)
    n_folds = int(n_folds)
    if n_folds < 2:
        raise ValueError("n_folds must be at least 2")
    for (cls, name) in ((False, "controls"), (True, "patients")):
        if int((labels == cls).sum()) < n_folds:
            raise ValueError("%d %s cannot be spread over %d folds" % (int((labels == cls).sum()), name, n_folds))
    rng = np.random.RandomState(seed)
    fold = np.empty(labels.size, dtype=np.int64)
    start = 0
    for cls in (False, True):
        idx = np.flatnonzero(labels == cls)
        idx = idx[rng.permutation(idx.size)]
        fold[idx] = (start + np.arange(idx.size)) % n_folds
        start += idx.size
    return fold


def cross_validate(corr, labels, n_folds=5, model=None, seed=0, fit_options=None, prior_patient=None, streams=None):
    """
    Stratified k-fold cross-validation of the two-group classifier
    (``UnsharedRegionFit.classify_subjects``): every fold is fitted on the
    other folds' subjects and classifies its own.

    Parameters
    ----------
    corr : (C, S) array or CUDA tensor
        Correlations of ALL subjects, one column per subject.
    labels : (S,) bool
        True for patients, False for controls.
    n_folds, seed
        Folds of :func:`stratified_folds`.
    model, fit_options, streams
        As for :func:`permutation_sweep` (one GPU; the folds are the replicas).
    prior_patient : float or None
        Prior probability of the patient group; None: each fold's training proportion.

    Returns
    -------
    dict with, per subject in column order, ``fold``, ``log_odds``, ``p_patient``,
    ``control_loglik`` and ``patient_elbo`` ((S,) arrays), and ``folds``: per fold
    the summary of its fit (fitted parameters, energy trace) with its final
    ``free_energy``.
    """
    labels = np.asarray(labels, dtype=bool).reshape(-1)
    fold = stratified_folds(labels, n_folds, seed)
    dev = _dev.device()
    corr_dev = corr if torch.is_tensor(corr) else torch.from_numpy(np.ascontiguousarray(corr, dtype=np.float64))
    corr_dev = corr_dev.to(dev, torch.float64)
    if corr_dev.dim() != 2 or int(corr_dev.shape[1]) != labels.size:
        raise ValueError("corr must be (C, S) with S = %d labels (got shape %s)" % (labels.size, tuple(corr_dev.shape)))
    model = UnsharedRegionModel() if model is None else model
    shared = None
    if not (fit_options or {}).get("update_mu_sigma"):
        shared = SharedPlanes(corr_dev, model, missing=(fit_options or {}).get("missing", "reject"))

    def run_one(i):
        train = fold != i
        con = torch.from_numpy(np.flatnonzero(train & ~labels)).to(dev)
        pat = torch.from_numpy(np.flatnonzero(train & labels)).to(dev)
        fit = UnsharedRegionFit()
        fit.model = copy.deepcopy(model)
        _configure(fit, fit_options)
        if shared is not None:
            fit.set_shared_inputs(shared, con, pat)
        else:
            fit.b = corr_dev.index_select(1, con)
            fit.bt = corr_dev.index_select(1, pat)
        fit.run()
        held = np.flatnonzero(fold == i)
        s = fit.classify_subjects(corr_dev.index_select(1, torch.from_numpy(held).to(dev)), prior_patient)
        return dict(held=held, scores=s, summary=dict(_summary(fit), free_energy=float(fit.energy[-1])))

    results = _run_replicas(list(range(n_folds)), run_one, default_streams() if streams is None else int(streams))
    out = dict(fold=fold, folds=[results[i]["summary"] for i in range(n_folds)])
    for name in ("log_odds", "p_patient", "control_loglik", "patient_elbo"):
        v = np.empty(labels.size, dtype=np.float64)
        for i in range(n_folds):
            v[results[i]["held"]] = getattr(results[i]["scores"], name)
        out[name] = v
    return out


def permutation_p_value(results, statistic=lambda r: -r["energy"][-1]):
    """One-sided permutation p-value of the observed labelling (replica 0): the
    share of labellings whose statistic is at least the observed one (the
    default statistic is the negative free energy, i.e. the evidence bound)."""
    obs = statistic(results[0])
    vals = [statistic(results[i]) for i in sorted(results)]
    return float(np.mean([v >= obs for v in vals]))


def restart_sweep(b, bt, n_restarts, model=None, seed=0, jitter=0.5, fit_options=None, rank=0, world=1,
                  group=None, gather=True):
    """
    Random restarts: replica 0 starts from ``model``; replica i > 0 from a copy
    whose (pi, eta, epsilon) are moved in logit space by N(0, jitter^2) draws of
    ``RandomState(seed + i)``.  Returns the summaries and the index of the
    replica with the lowest final free energy.
    """
    dev = _dev.device()
    to_dev = lambda a: (a if torch.is_tensor(a) else torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64))).to(dev, torch.float64)
    (b_dev, bt_dev) = (to_dev(b), to_dev(bt))
    model = UnsharedRegionModel() if model is None else model
    results = {}
    for i in replica_indices(n_restarts + 1, rank, world):
        m = copy.deepcopy(model)
        if i > 0:
            rng = np.random.RandomState(seed + i)
            for name in ("pi", "eta", "epsilon"):
                x = float(getattr(m, name))
                z = np.log(x / (1.0 - x)) + jitter * rng.normal()
                setattr(m, name, float(min(max(1.0 / (1.0 + np.exp(-z)), 1e-4), 1 - 1e-4)))
        fit = UnsharedRegionFit()
        fit.model = m
        _configure(fit, fit_options)
        (fit.b, fit.bt) = (b_dev, bt_dev)
        fit.run()
        results[i] = _summary(fit)
        del fit
    results = _gather(results, group) if gather else results
    best = min(results, key=lambda i: results[i]["energy"][-1])
    return results, best
