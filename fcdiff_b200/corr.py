"""
Region time series -> subject correlations in the layout ``fcdiff.fit`` consumes.

New stage (the reference's inputs *are* the correlations, fcdiff/fit.py:20-23;
SURVEY 8 a11): per subject the (N, T) time series are standardised, the Gram
matrix R = Z Z^T is formed on the GPU and its strict lower triangle is written
in ``util`` edge order to column s of a (C, S) float64 matrix -- Fisher-z
transformed (``arctanh``) by default.  Oracle: ``numpy.corrcoef`` +
``numpy.arctanh`` (``oracle/iar_oracle.py:corr_fisherz``).
"""
import numpy as np
import torch

from . import _dev, _lib
from .util import N_to_C


def correlations_device(ts_dev, fisher=True, out=None, s0=0, missing=False):
    """ts_dev: float32 CUDA tensor (S, N, T).  Returns / fills a float64 CUDA
    tensor (C, pitch) with columns [s0, s0 + S) written.  ``missing``: see
    :func:`correlations`."""
    lib = _lib.load()
    (S, N, T) = ts_dev.shape
    C = N_to_C(N)
    if out is None:
        out = _dev.empty((C, s0 + S))
    pitch = out.shape[1]
    zws = torch.empty(lib.fcd_corr_workspace_bytes(S, N, T), dtype=torch.uint8, device=ts_dev.device)
    _lib.check(lib.fcd_corr_fisherz(_dev.ptr(ts_dev), S, N, T, _dev.ptr(out), pitch, s0, 1 if fisher else 0,
                                    _dev.ptr(zws), _dev.stream()), "fcd_corr_fisherz")
    if missing:
        _lib.check(lib.fcd_corr_mark_missing(_dev.ptr(ts_dev), S, N, T, _dev.ptr(out), pitch, s0, _dev.stream()),
                   "fcd_corr_mark_missing")
    return out


def correlations(ts, fisher=True, missing=False):
    """
    Computes subject correlations from region time series.

    Arguments
    ---------
    ts : :class:`numpy.ndarray`, (S, N, T), float
        Region time series of S subjects, N regions, T time points.
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
        clip (a NaN sample).

    Returns
    -------
    :class:`numpy.ndarray`, (C, S), float64 -- connection-major, subject-minor.
    """
    ts_dev = _dev.upload(np.asarray(ts), np.float32)
    return _dev.download(correlations_device(ts_dev, fisher=fisher, missing=missing))
