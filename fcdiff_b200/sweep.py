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
import collections
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


def _summary(fit, q1=None):
    """``q1``: ``np.exp(fit._lq_R[:, :, 1])`` when the caller has it already."""
    m = fit.model
    q1 = np.exp(fit._lq_R[:, :, 1]) if q1 is None else q1
    return dict(energy=list(fit.energy), pi=float(m.pi), eta=float(m.eta), epsilon=float(m.epsilon),
                gamma=np.asarray(m.gamma, dtype=np.float64).copy(), mu=np.asarray(m.mu, dtype=np.float64).copy(),
                sigma=np.asarray(m.sigma, dtype=np.float64).copy(), iterations=len(fit.energy) - 1,
                expected_anomalous_regions=float(q1.sum()))


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
    results = _permutation_replicas(corr, labels, n_permutations, model, seed, fit_options, rank, world,
                                    shared_planes, streams)
    return _gather(results, group) if gather else results


def _permutation_replicas(corr, labels, n_permutations, model, seed, fit_options, rank, world, shared_planes,
                          streams, write_row=None):
    """This rank's replicas of :func:`permutation_sweep`, not gathered.  ``write_row(fit, i, q1)``, when given,
    runs after replica i's fit, on the stream the fit ran on, with ``q1 = np.exp(fit._lq_R[:, :, 1])``."""
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
        if write_row is None:
            return _summary(fit)
        q1 = np.exp(fit._lq_R[:, :, 1])                # one pass for the row and the summary
        write_row(fit, i, q1)
        return _summary(fit, q1)

    return _run_replicas(replica_indices(n_permutations + 1, rank, world), run_one,
                         default_streams(world) if streams is None else int(streams))


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


def _check_families(K, families):
    """[(start, stop)] of ``families`` (default: one family of all K columns): non-empty, inside [0, K) and
    disjoint."""
    if families is None:
        return [(0, K)]
    out = []
    for fam in families:
        (a, b) = (int(fam[0]), int(fam[1]))
        if not 0 <= a < b <= K:
            raise ValueError("family (%d, %d) is not a non-empty range of the %d columns" % (a, b, K))
        out.append((a, b))
    if not out:
        raise ValueError("families holds no range")
    s = sorted(out)
    for (x, y) in zip(s[:-1], s[1:]):
        if y[0] < x[1]:
            raise ValueError("families (%d, %d) and (%d, %d) overlap" % (x + y))
    return out


def maxt_pvalues(stats, families=None):
    """
    Permutation p-values of every column of a statistics matrix, uncorrected and with family-wise error control
    by the Westfall-Young step-down max-T procedure (Westfall & Young 1993, algorithm 4.1).

    One-sided: large values are evidence against H0.  Within a family F of columns, with T = ``stats``:
    ``p[k] = #{r : T[r,k] >= T[0,k]} / R1`` (row 0 is counted, so p >= 1 / R1), and with sigma ordering F
    ascending by ``(T[0,k], k)``, ``count[j] = #{r : max_{i <= j} T[r,sigma(i)] >= T[0,sigma(j)]}`` and
    ``p_fwer[sigma(j)] = max_{i >= j} count[i] / R1`` -- the step-down in descending order, written with prefix
    maxima.  Tied observed values get equal p_fwer, and p_fwer >= p.  The rows must be exchangeable under H0
    (relabelled data).  The counting runs on the GPU (``fcd_maxt_counts``, csrc/fcd_permutation.cu); the counts
    are integers, so the result is exact.

    Parameters
    ----------
    stats : (R1, K) CUDA tensor or host array
        Row 0 the observed statistics, rows 1.. those of R1 - 1 relabellings.  Must be finite.
    families : sequence of (start, stop) or None
        Disjoint column ranges, each a family of its own; default: one family of all K columns.

    Returns
    -------
    (p, p_fwer) : (K,) float64 host arrays; NaN in columns outside every family.  Besides ``stats`` on the
    device, the counting takes 8 R1 (Kf + Kf / 512) bytes of scratch, Kf the widest family.
    """
    if torch.is_tensor(stats):
        shape = tuple(stats.shape)
    else:
        stats = np.asarray(stats, dtype=np.float64)
        shape = stats.shape
    if len(shape) != 2:
        raise ValueError("stats must be (R1, K) (got shape %s)" % (shape,))
    (R1, K) = (int(shape[0]), int(shape[1]))
    if R1 < 1 or K < 1:
        raise ValueError("stats must have at least one row and one column (got shape %s)" % (shape,))
    fams = _check_families(K, families)
    if torch.is_tensor(stats):
        ok = torch.isfinite(stats).all(dim=0).cpu().numpy()          # one device reduction
    else:
        ok = np.isfinite(stats).all(axis=0)
    if not ok.all():
        raise ValueError("stats holds a NaN or infinite value in column %d" % int(np.flatnonzero(~ok)[0]))

    import ctypes
    from . import _lib
    lib = _lib.load()
    if torch.is_tensor(stats):
        T = stats.to(_dev.device(), torch.float64).contiguous()
    else:
        T = _dev.upload(stats)
    obs = _dev.download(T[0])
    width = max(b - a for (a, b) in fams)
    nws = int(lib.fcd_maxt_ws_bytes(R1, width)) // 8
    if nws < 1:
        raise ValueError("stats of shape %s exceed the counting kernel's limits" % (shape,))
    ws = _dev.empty((nws,))
    (p, p_fwer) = (np.full(K, np.nan), np.full(K, np.nan))
    for (a, b) in fams:
        sigma = np.lexsort((np.arange(b - a), obs[a:b]))
        order = _dev.upload(sigma + a, np.int64)
        (cu, cs) = (_dev.empty((b - a,), torch.int64), _dev.empty((b - a,), torch.int64))
        _lib.check(lib.fcd_maxt_counts(_dev.ptr(T), R1, K, K, _dev.ptr(order), a, b, _dev.ptr(cu), _dev.ptr(cs),
                                       _dev.ptr(ws), _dev.stream()), "fcd_maxt_counts")
        p[a:b] = _dev.download(cu) / R1
        p_fwer[a + sigma] = np.maximum.accumulate(_dev.download(cs)[::-1])[::-1] / R1
    return p, p_fwer


# what permutation_inference returns
PermutationInference = collections.namedtuple(
    "PermutationInference", "region_rate region_p region_p_fwer region_q connection_rate connection_p "
                            "connection_p_fwer connection_q statistics replica_index replicas")


def permutation_inference(corr, labels, n_permutations, model=None, seed=0, fit_options=None, connections=True,
                          rank=0, world=1, group=None, gather=True, shared_planes=True, streams=None):
    """
    Which regions, and which connections, are anomalous in the patient group more often than chance: per-replica
    anomaly rates of the permutation sweep turned into permutation p-values with family-wise error control.

    The replicas -- labellings, sharding, streams, shared planes -- are those of :func:`permutation_sweep` with
    the same arguments.  After each fit, one row of statistics is written on the device:

    * region n: ``region_rate[n] = mean_u q_R[n, u, anomalous]``, the expected share of patients in whom region
      n is anomalous (``np.exp(fit._lq_R[:, :, 1]).mean(axis=1)``);
    * connection c: ``connection_rate[c]``, the ``anomalous_rate`` of ``fit.connection_posteriors(maps=False)``,
      written straight into the row.

    Under H0 (patients and controls have the same distribution) the labellings are exchangeable, and so are
    the rows.  The regions and the connections are two families, each with its own :func:`maxt_pvalues`:
    ``*_p`` uncorrected, ``*_p_fwer`` step-down max-T (strong family-wise error control within the family),
    ``*_q`` Benjamini-Hochberg adjusted ``*_p`` within the family (``scipy.stats.false_discovery_control``; they
    control the false discovery rate when the p-values are independent or positively regression dependent
    on the subset of true nulls, PRDS).

    Parameters
    ----------
    corr, labels, n_permutations, model, seed, fit_options, rank, world, group, shared_planes, streams
        As for :func:`permutation_sweep`.  ``labels`` needs at least one control and one patient;
        ``n_permutations = 0`` gives every p-value 1.
    connections : bool
        Keep the connection statistics (default).  False keeps the N region columns only.
    gather : bool
        With ``world > 1`` the ranks' rows are gathered (``torch.distributed.all_gather_into_tensor``; an
        initialised process group of ``world`` ranks is required), and every rank computes the same p-values.
        False: the p-value fields are None and ``statistics`` / ``replica_index`` hold this rank's rows, to be
        stacked in replica order and passed to :func:`maxt_pvalues`.

    Returns
    -------
    PermutationInference(region_rate, region_p, region_p_fwer, region_q, connection_rate, connection_p,
    connection_p_fwer, connection_q, statistics, replica_index, replicas):
        the ``*_rate`` fields are the observed statistics, (N,) and (C,) float64 (None on a rank that does not
        hold replica 0); the p-value fields (N,) and (C,) float64; the connection fields are None without
        ``connections``.  ``statistics`` is the (rows, N [+ C]) float64 CUDA tensor, row j that of replica
        ``replica_index[j]``; ``replicas`` the summaries :func:`permutation_sweep` returns.

    Memory: ``statistics`` takes 8 (n_permutations + 1)(N + C) bytes on the device -- 642 MB at 400 regions and
    1000 permutations, 4.0 GB at 1000 regions -- and the counting as much again, for the connection family.
    """
    import torch.distributed as dist
    from .util import C_to_N
    labels = np.asarray(labels, dtype=bool).reshape(-1)
    n_permutations = int(n_permutations)
    if n_permutations < 0:
        raise ValueError("n_permutations must be >= 0 (got %d)" % n_permutations)
    if not labels.any() or labels.all():
        raise ValueError("labels must hold at least one control and one patient")
    shape = tuple(corr.shape) if torch.is_tensor(corr) else np.shape(corr)
    if len(shape) != 2 or int(shape[1]) != labels.size:
        raise ValueError("corr must be (C, S) with S = %d labels (got shape %s)" % (labels.size, shape))
    C = int(shape[0])
    N = C_to_N(C)
    if N % 1 != 0 or C < 1:
        raise ValueError("Number of connections (%u) must be a triangular number." % C)
    N = int(N)
    (rank, world) = (int(rank), int(world))
    if world < 1 or not 0 <= rank < world:
        raise ValueError("rank %d of world %d" % (rank, world))
    active = dist.is_available() and dist.is_initialized()
    if gather and world > 1:
        if not active:
            raise ValueError("gathering the statistics of world > 1 ranks needs an initialised process group")
        if dist.get_world_size(group) != world:
            raise ValueError("world = %d, but the process group has %d ranks" % (world, dist.get_world_size(group)))

    R1 = n_permutations + 1
    idx = replica_indices(R1, rank, world)
    row_of = {i: j for (j, i) in enumerate(idx)}
    K = N + (C if connections else 0)
    stats = _dev.empty((len(idx), K))                # on the caller's stream, before the workers start

    def write_row(fit, i, q1):
        j = row_of[i]
        stats[j, :N].copy_(torch.from_numpy(q1.mean(axis=1)))
        if connections:
            fit._connection_rate_into(stats[j, N:])

    results = _permutation_replicas(corr, labels, n_permutations, model, seed, fit_options, rank, world,
                                    shared_planes, streams, write_row)
    index = np.asarray(idx, dtype=np.int64)
    if not gather:
        obs = _dev.download(stats[0]) if 0 in row_of else None
        return PermutationInference(None if obs is None else obs[:N], None, None, None,
                                    None if obs is None or not connections else obs[N:], None, None, None,
                                    stats, index, results)
    if world > 1:
        pad = -(-R1 // world)
        local = _dev.zeros((pad, K))
        local[:len(idx)].copy_(stats)
        out = _dev.empty((world * pad, K))
        dist.all_gather_into_tensor(out, local, group=group)
        src = torch.tensor([(i % world) * pad + i // world for i in range(R1)], dtype=torch.int64,
                           device=out.device)
        (stats, index) = (out.index_select(0, src), np.arange(R1, dtype=np.int64))
        results = _gather(results, group)
    import scipy.stats
    fams = [(0, N)] + ([(N, N + C)] if connections else [])
    (p, p_fwer) = maxt_pvalues(stats, fams)
    obs = _dev.download(stats[0])
    fields = []
    for (a, b) in ((0, N), (N, N + C)):
        if b > K:
            fields += [None] * 4
        else:
            fields += [obs[a:b], p[a:b], p_fwer[a:b], scipy.stats.false_discovery_control(p[a:b], method="bh")]
    return PermutationInference(*fields, statistics=stats, replica_index=index, replicas=results)


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
