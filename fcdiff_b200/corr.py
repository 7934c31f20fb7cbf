"""
Region time series -> subject correlations in the layout ``fcdiff.fit`` consumes.

New stage (the reference's inputs *are* the correlations, fcdiff/fit.py:20-23;
SURVEY 8 a11): per subject the (N, T) time series are standardised, the Gram
matrix R = Z Z^T is formed on the GPU and its strict lower triangle is written
in ``util`` edge order to column s of a (C, S) float64 matrix -- Fisher-z
transformed (``arctanh``) by default.  Oracle: ``numpy.corrcoef`` +
``numpy.arctanh`` (``oracle/iar_oracle.py:corr_fisherz``).

Cleaned time series (``sample_mask`` / ``confounds``, ``fcd_corr_fisherz_clean``): frames can be censored
per subject, subjects can differ in length, and nuisance regressors are projected out of every region on
the GPU before the correlations.  Oracle: ``oracle/clean.py``.

Partial correlations (``kind="partial"``, ``fcd_corr_partial``): per subject the cleaned rows in fp64, a
Ledoit-Wolf shrunk correlation matrix and its inverse P on the GPU, r_nm = -P_nm / sqrt(P_nn P_mm).
Oracle: ``oracle/partial.py``.
"""
import numpy as np
import torch

from . import _dev, _lib
from .util import N_to_C


MAX_CONFOUNDS = 64
KINDS = ("pearson", "partial")


def check_kind(kind, shrinkage):
    """Validates ``kind`` and ``shrinkage`` on the host; returns the shrinkage the library takes (-1.0 for
    Ledoit-Wolf).  Raises ``ValueError`` for an unknown kind or a shrinkage that is neither
    ``"ledoit-wolf"`` nor a number in [0, 1]."""
    if kind not in KINDS:
        raise ValueError("kind: expected one of %s, got %r" % (KINDS, kind))
    if isinstance(shrinkage, str):
        if shrinkage != "ledoit-wolf":
            raise ValueError("shrinkage: expected \"ledoit-wolf\" or a number in [0, 1], got %r" % shrinkage)
        return -1.0
    d = float(shrinkage)
    if not 0.0 <= d <= 1.0:
        raise ValueError("shrinkage: %r outside [0, 1]" % (shrinkage,))
    return d


def _check_not_singular(n, N, K, d):
    """shrinkage = 0 leaves the sample correlation matrix, singular when a subject keeps n_s <= N + K frames."""
    if d == 0.0 and (n <= N + K).any():
        s = int(np.argmax(n <= N + K))
        raise ValueError("shrinkage=0: subject %d keeps %d frames, its correlation matrix of %d regions after %d "
                         "confounds is singular (needs more than %d)" % (s, int(n[s]), N, K, N + K))


def pack_clean(ts, sample_mask=None, confounds=None):
    """
    Packs and validates the inputs of a cleaned correlation run on the host (no device work).

    ``ts`` is an (S, N, T) array or a list of (N, T_s) arrays; ``sample_mask`` None, an (S, T) bool array or a
    list of (T_s,) bool arrays (True: the frame is kept); ``confounds`` None, an (S, T, K) array or a list of
    (T_s, K) arrays.  Returns ``(ts, keep, conf)``: ts (S, N, T_max) float32 zero-padded, keep (S, T_max)
    uint8 (frame t of subject s is kept iff t < T_s and its mask keeps it), conf (S, T_max, K) float64
    zero-padded, or None when ``confounds`` is None.  Raises ``ValueError`` for mismatched shapes, K > 64,
    a non-finite confound on a kept frame, or a subject with fewer than K + 2 kept frames.
    """
    if isinstance(ts, (list, tuple)):
        subjects = [np.asarray(x) for x in ts]
        if not subjects:
            raise ValueError("ts: no subjects")
        if any(x.ndim != 2 for x in subjects):
            raise ValueError("ts: every subject must be an (N, T_s) array")
        N = subjects[0].shape[0]
        if any(x.shape[0] != N for x in subjects):
            raise ValueError("ts: subjects differ in regions: %s" % sorted({x.shape[0] for x in subjects}))
        lengths = np.array([x.shape[1] for x in subjects], dtype=np.int64)
        packed = np.zeros((len(subjects), N, int(lengths.max())), dtype=np.float32)
        for (s, x) in enumerate(subjects):
            packed[s, :, :x.shape[1]] = x
    else:
        packed = np.ascontiguousarray(np.asarray(ts), dtype=np.float32)
        if packed.ndim != 3:
            raise ValueError("ts: expected (S, N, T) or a list of (N, T_s), got shape %s" % (packed.shape,))
        lengths = np.full(packed.shape[0], packed.shape[2], dtype=np.int64)
    (S, N, T) = packed.shape
    if N < 2 or T < 2:
        raise ValueError("ts: need N >= 2 regions and T >= 2 time points, got (%d, %d)" % (N, T))

    def ragged(a, name, tail):
        """(S, T_max) + tail array from an array or a list of (T_s,) + tail arrays, zero-padded."""
        if isinstance(a, (list, tuple)):
            if len(a) != S:
                raise ValueError("%s: %d subjects, ts has %d" % (name, len(a), S))
            out = None
            for (s, x) in enumerate(a):
                x = np.asarray(x)
                if x.ndim != 1 + len(tail) or x.shape[0] != lengths[s] or (tail and x.shape[1:] != tail):
                    raise ValueError("%s: subject %d has shape %s, expected %s" % (
                        name, s, x.shape, (int(lengths[s]),) + tail))
                if out is None:
                    out = np.zeros((S, T) + tail, dtype=x.dtype)
                out[s, :x.shape[0]] = x
            return out
        a = np.asarray(a)
        if a.shape[:2] != (S, T) or a.ndim != 2 + len(tail) or (tail and a.shape[2:] != tail):
            raise ValueError("%s: shape %s, expected %s" % (name, a.shape, (S, T) + tail))
        return a

    keep = np.arange(T)[None, :] < lengths[:, None]
    if sample_mask is not None:
        m = ragged(sample_mask, "sample_mask", ())
        if m.dtype != np.bool_:
            raise ValueError("sample_mask: expected bool, got %s" % m.dtype)
        keep &= m
    conf = None
    K = 0
    if confounds is not None:
        if isinstance(confounds, (list, tuple)):
            first = np.asarray(confounds[0]) if len(confounds) else np.zeros((0, 0))
            if first.ndim != 2:
                raise ValueError("confounds: every subject must be a (T_s, K) array")
            K = first.shape[1]
        else:
            K = np.asarray(confounds).shape[-1] if np.asarray(confounds).ndim == 3 else -1
            if K < 0:
                raise ValueError("confounds: expected (S, T, K), got shape %s" % (np.asarray(confounds).shape,))
        if K > MAX_CONFOUNDS:
            raise ValueError("confounds: K = %d > %d columns" % (K, MAX_CONFOUNDS))
        conf = np.ascontiguousarray(ragged(confounds, "confounds", (K,)), dtype=np.float64)
        bad = ~np.isfinite(conf).all(axis=2) & keep
        if bad.any():
            (s, t) = np.argwhere(bad)[0]
            raise ValueError("confounds: non-finite value on kept frame %d of subject %d" % (t, s))
        if K == 0:
            conf = None
    n = keep.sum(axis=1)
    if (n < K + 2).any():
        s = int(np.argmax(n < K + 2))
        raise ValueError("subject %d keeps %d frames; %d confounds need at least %d" % (s, n[s], K, K + 2))
    return packed, keep.astype(np.uint8), conf


def correlations_device(ts_dev, fisher=True, out=None, s0=0, missing=False, sample_mask=None, confounds=None,
                        rank=None, kind="pearson", shrinkage="ledoit-wolf", shrinkage_out=None):
    """ts_dev: float32 CUDA tensor (S, N, T).  Returns / fills a float64 CUDA
    tensor (C, pitch) with columns [s0, s0 + S) written.  ``missing``: see
    :func:`correlations`.  ``sample_mask`` ((S, T) bool) and ``confounds``
    ((S, T, K) float64), as arrays or CUDA tensors, select the cleaned path
    (:func:`correlations`; checked as :func:`pack_clean` does); ``rank``: an
    optional (S,) int32 CUDA tensor that receives the confounds kept per subject.
    ``kind`` / ``shrinkage``: see :func:`correlations`; ``shrinkage_out``: an
    optional (S,) float64 CUDA tensor that receives the shrinkage of each subject
    (partial correlations only)."""
    d = check_kind(kind, shrinkage)
    lib = _lib.load()
    (S, N, T) = ts_dev.shape
    C = N_to_C(N)
    if out is None:
        out = _dev.empty((C, s0 + S))
    pitch = out.shape[1]
    if kind == "pearson" and shrinkage_out is not None:
        raise ValueError("shrinkage_out: only kind=\"partial\" has a shrinkage")
    if kind == "pearson" and sample_mask is None and confounds is None:
        zws = torch.empty(lib.fcd_corr_workspace_bytes(S, N, T), dtype=torch.uint8, device=ts_dev.device)
        _lib.check(lib.fcd_corr_fisherz(_dev.ptr(ts_dev), S, N, T, _dev.ptr(out), pitch, s0, 1 if fisher else 0,
                                        _dev.ptr(zws), _dev.stream()), "fcd_corr_fisherz")
        if missing:
            _lib.check(lib.fcd_corr_mark_missing(_dev.ptr(ts_dev), S, N, T, _dev.ptr(out), pitch, s0,
                                                 _dev.stream()), "fcd_corr_mark_missing")
        return out
    keep = None
    if sample_mask is not None:
        keep = torch.as_tensor(sample_mask, device=ts_dev.device)
        if keep.dtype != torch.bool or tuple(keep.shape) != (S, T):
            raise ValueError("sample_mask: expected (S, T) = %s bool, got %s %s" % ((S, T), tuple(keep.shape),
                                                                                  keep.dtype))
        keep = keep.to(torch.uint8).contiguous()
    conf = None
    K = 0
    if confounds is not None:
        conf = torch.as_tensor(confounds, device=ts_dev.device).to(torch.float64).contiguous()
        if conf.dim() != 3 or tuple(conf.shape[:2]) != (S, T):
            raise ValueError("confounds: expected (S, T, K) with (S, T) = %s, got %s" % ((S, T), tuple(conf.shape)))
        K = int(conf.shape[2])
        if K > MAX_CONFOUNDS:
            raise ValueError("confounds: K = %d > %d columns" % (K, MAX_CONFOUNDS))
        kept = keep.bool() if keep is not None else torch.ones((S, T), dtype=torch.bool, device=ts_dev.device)
        if bool((~torch.isfinite(conf).all(dim=2) & kept).any()):
            raise ValueError("confounds: non-finite value on a kept frame")
        if K == 0:
            conf = None
    n = keep.sum(dim=1) if keep is not None else torch.full((S,), T, device=ts_dev.device)
    if bool((n < K + 2).any()):
        raise ValueError("a subject keeps fewer than K + 2 = %d frames" % (K + 2))
    if kind == "partial":
        _check_not_singular(n.cpu().numpy(), N, K, d)
        if shrinkage_out is not None and (shrinkage_out.dtype != torch.float64 or tuple(shrinkage_out.shape) != (S,)
                                          or not shrinkage_out.is_contiguous()):
            raise ValueError("shrinkage_out: expected a contiguous (%d,) float64 tensor" % S)
        status = torch.empty((S,), dtype=torch.int32, device=ts_dev.device)
        zws = torch.empty(lib.fcd_corr_partial_workspace_bytes(S, N, T, K), dtype=torch.uint8, device=ts_dev.device)
        _lib.check(lib.fcd_corr_partial(_dev.ptr(ts_dev), S, N, T, _dev.ptr(keep), _dev.ptr(conf), K, d, _dev.ptr(out),
                                        pitch, s0, 1 if fisher else 0, 1 if missing else 0, _dev.ptr(rank),
                                        _dev.ptr(shrinkage_out), _dev.ptr(status), _dev.ptr(zws), _dev.stream()),
                   "fcd_corr_partial")
        bad = torch.nonzero(status).flatten().tolist()
        if bad:
            raise ValueError("partial correlations: the shrunk correlation matrix of subject(s) %s is singular to "
                             "working precision (their columns are NaN); use a shrinkage > 0" % bad)
        return out
    zws = torch.empty(lib.fcd_corr_clean_workspace_bytes(S, N, T, K), dtype=torch.uint8, device=ts_dev.device)
    _lib.check(lib.fcd_corr_fisherz_clean(_dev.ptr(ts_dev), S, N, T, _dev.ptr(keep), _dev.ptr(conf), K, _dev.ptr(out),
                                          pitch, s0, 1 if fisher else 0, 1 if missing else 0, _dev.ptr(rank),
                                          _dev.ptr(zws), _dev.stream()), "fcd_corr_fisherz_clean")
    return out


def correlations(ts, fisher=True, missing=False, sample_mask=None, confounds=None, kind="pearson",
                 shrinkage="ledoit-wolf", return_shrinkage=False):
    """
    Computes subject correlations from region time series.

    Arguments
    ---------
    ts : :class:`numpy.ndarray`, (S, N, T), float, or a list of (N, T_s) arrays
        Region time series of S subjects, N regions, T time points.  A list
        may hold subjects of different lengths T_s (cleaned path).
    fisher : bool
        Apply the Fisher z-transform (default) or return Pearson r clipped to
        [-1, 1] (what the reference's model is specified on, doc/methods.rst:163-165).
    missing : bool
        Mark the regions without a usable time series in a subject -- a
        non-finite sample (a parcel outside the field of view, a dropped-out
        signal) or zero variance -- as not observed: all their connections of
        that subject are NaN, for a fit with ``missing="marginalize"``.  Every
        other entry is the same as with ``missing=False``, which gives such a
        region r = 0 against every other region (zero variance) or the negative
        clip (a NaN sample).  On the cleaned path only kept frames count, a
        region explained by the confounds (residual sum of squares at most
        2^-40 of its centred one) is also unusable, and an unusable region
        gets r = 0 with ``missing=False``.
    sample_mask : None, (S, T) bool array or list of (T_s,) bool arrays
        Frames to keep (True) per subject; a censored (scrubbed) frame is left
        out of the correlations, whatever its samples hold (NaN included).
    confounds : None, (S, T, K) array or list of (T_s, K) arrays, K <= 64
        Nuisance regressors per frame (motion parameters, WM / CSF / global
        signals, trends).  Each region is cleared of them and of a constant
        over the kept frames on the GPU: r is the partial correlation given
        the confounds.  Collinear columns are dropped.
    kind : ``"pearson"`` (default) or ``"partial"``
        ``"partial"``: the partial correlation of every two regions given all
        other regions (and the confounds and a constant), as nilearn's
        ``ConnectivityMeasure(kind="partial correlation")``: per subject the
        cleaned rows are scaled to unit variance (1/n_s normalisation over its
        n_s kept frames), their correlation matrix R is shrunk to
        Sigma = (1 - delta) R + delta mu I (mu = tr R / N) and inverted in
        fp64 on the GPU, r_nm = -P_nm / sqrt(P_nn P_mm) with P = Sigma^-1.
        Unusable regions (as above) are left out of their subject's problem.
        Partial correlations are smaller in magnitude than full ones: set the
        fit's ``model.mu`` / ``model.sigma`` or use ``update_mu_sigma=True``.
    shrinkage : ``"ledoit-wolf"`` (default) or a float in [0, 1]
        delta of ``kind="partial"``: the Ledoit-Wolf estimate of
        ``sklearn.covariance.ledoit_wolf`` on the unit-variance rows (which
        counts n_s samples; the K + 1 fitted confound columns are not
        subtracted), or a fixed value.  0 needs more than N + K kept frames per
        subject; a subject whose shrunk matrix is still singular to working
        precision raises ``ValueError``.
    return_shrinkage : bool
        Also return the (S,) delta of every subject (``kind="partial"``).

    With ``sample_mask`` and ``confounds`` both None and an array ``ts`` this
    is the plain path (``fcd_corr_fisherz``); otherwise the inputs are packed
    and checked by :func:`pack_clean` and the cleaned path runs.

    Returns
    -------
    :class:`numpy.ndarray`, (C, S), float64 -- connection-major, subject-minor;
    with ``return_shrinkage`` the pair (correlations, (S,) float64 delta).
    """
    d = check_kind(kind, shrinkage)
    if return_shrinkage and kind != "partial":
        raise ValueError("return_shrinkage: only kind=\"partial\" has a shrinkage")
    if kind == "partial":
        (packed, keep, conf) = pack_clean(ts, sample_mask, confounds)
        _check_not_singular(keep.sum(axis=1), packed.shape[1], 0 if conf is None else conf.shape[2], d)
        delta = _dev.empty((packed.shape[0],))
        out = _dev.download(correlations_device(
            _dev.upload(packed, np.float32), fisher=fisher, missing=missing,
            sample_mask=_dev.upload(keep.astype(np.bool_), np.bool_),
            confounds=_dev.upload(conf, np.float64) if conf is not None else None, kind=kind, shrinkage=shrinkage,
            shrinkage_out=delta))
        return (out, _dev.download(delta)) if return_shrinkage else out
    if sample_mask is None and confounds is None and not isinstance(ts, (list, tuple)):
        ts_dev = _dev.upload(np.asarray(ts), np.float32)
        return _dev.download(correlations_device(ts_dev, fisher=fisher, missing=missing))
    (packed, keep, conf) = pack_clean(ts, sample_mask, confounds)
    keep_dev = _dev.upload(keep.astype(np.bool_), np.bool_)
    conf_dev = _dev.upload(conf, np.float64) if conf is not None else None
    return _dev.download(correlations_device(_dev.upload(packed, np.float32), fisher=fisher, missing=missing,
                                             sample_mask=keep_dev, confounds=conf_dev))
