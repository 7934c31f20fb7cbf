"""
Input adapters: region time series on disk -> the (C, H) / (C, U) correlation
matrices ``fcdiff.fit`` consumes (SURVEY 8f item 3).  The reference has no I/O
at all (README.rst:19-28): its inputs *are* the correlations (fcdiff/fit.py:20-23).

One file per subject holding an (N regions x T time points) table, or (T x N) with
``time_major=True``:

* ``.npy``                      -- numpy array;
* ``.csv`` / ``.tsv`` / ``.txt`` -- delimited text (``#`` comments, optional header line);
* ``.nii`` / ``.nii.gz``        -- parcellated NIfTI time series via nibabel (not bundled:
                                   a clear ImportError if it is missing).

Only parsing happens on the host; standardisation, the Gram matrices and the
Fisher z-transform run on the GPU (``fcdiff_b200.corr``, K1).
"""
import os

import numpy as np

from . import corr


def load_subject(path, time_major=False):
    """(N, T) float32 time series of one subject."""
    ext = path.lower()
    if ext.endswith(".npy"):
        a = np.load(path)
    elif ext.endswith((".nii", ".nii.gz")):
        try:
            import nibabel
        except ImportError as e:        # pragma: no cover - optional dependency
            raise ImportError("reading %s needs nibabel, which is not installed" % path) from e
        a = np.asarray(nibabel.load(path).get_fdata())
        a = a.reshape(-1, a.shape[-1])                      # (regions, time)
    elif ext.endswith((".csv", ".tsv", ".txt")):
        delim = "\t" if ext.endswith(".tsv") else ("," if ext.endswith(".csv") else None)
        with open(path) as f:
            first = f.readline()
        skip = 0
        try:
            [float(tok) for tok in first.replace(",", " ").split() if tok]
        except ValueError:
            skip = 1                                        # header line
        a = np.loadtxt(path, delimiter=delim, skiprows=skip, comments="#", ndmin=2)
    else:
        raise ValueError("unsupported time-series file: %s" % path)
    a = np.asarray(a, dtype=np.float32)
    if a.ndim != 2:
        raise ValueError("%s: expected a 2-D table, got shape %s" % (path, a.shape))
    return np.ascontiguousarray(a.T if time_major else a)


def load_timeseries(paths, time_major=False):
    """(S, N, T) float32 from one file per subject; all subjects must share N and T
    (truncate or resample beforehand otherwise)."""
    subjects = [load_subject(p, time_major) for p in paths]
    shapes = {s.shape for s in subjects}
    if len(shapes) != 1:
        raise ValueError("subjects differ in (regions, time points): %s" % sorted(shapes))
    return np.stack(subjects, axis=0)


def correlations_from_files(control_paths, patient_paths, fisher=True, time_major=False, missing=False):
    """(b, bt): (C, H) and (C, U) float64 correlation matrices of the control and
    the patient group, ready for ``UnsharedRegionFit.b`` / ``.bt``.  ``missing``:
    regions without a usable time series in a subject give NaN connections
    (``corr.correlations``), for a fit with ``missing="marginalize"``."""
    ts = load_timeseries(list(control_paths) + list(patient_paths), time_major)
    c = corr.correlations(ts, fisher=fisher, missing=missing)
    H = len(control_paths)
    return np.ascontiguousarray(c[:, :H]), np.ascontiguousarray(c[:, H:])
