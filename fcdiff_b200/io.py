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

Cleaned inputs: ``load_timeseries_list`` keeps each subject's own length,
``load_confounds`` reads nuisance regressors (``.npy``, or a ``.tsv`` / ``.csv``
table with a header line such as fMRIPrep's confound files), and
``cleaned_correlations_from_files`` censors frames and regresses the confounds
out on the GPU before the correlations.
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


def correlations_from_files(control_paths, patient_paths, fisher=True, time_major=False, missing=False,
                            kind="pearson", shrinkage="ledoit-wolf"):
    """(b, bt): (C, H) and (C, U) float64 correlation matrices of the control and
    the patient group, ready for ``UnsharedRegionFit.b`` / ``.bt``.  ``missing``:
    regions without a usable time series in a subject give NaN connections
    (``corr.correlations``), for a fit with ``missing="marginalize"``.
    ``kind`` / ``shrinkage``: ``"partial"`` for partial correlations
    (``corr.correlations``)."""
    ts = load_timeseries(list(control_paths) + list(patient_paths), time_major)
    c = corr.correlations(ts, fisher=fisher, missing=missing, kind=kind, shrinkage=shrinkage)
    H = len(control_paths)
    return np.ascontiguousarray(c[:, :H]), np.ascontiguousarray(c[:, H:])


def load_timeseries_list(paths, time_major=False):
    """List of (N, T_s) float32 arrays, one per file; the subjects must share N but may differ in length."""
    subjects = [load_subject(p, time_major) for p in paths]
    regions = {s.shape[0] for s in subjects}
    if len(regions) > 1:
        raise ValueError("subjects differ in regions: %s" % sorted(regions))
    return subjects


def load_confounds(path, columns=None):
    """
    (T, K) float64 confounds of one subject.  ``.npy``: a (T, K) array (or (T,), read as one column),
    ``columns`` then indexes its columns.  ``.tsv`` / ``.csv``: a table with a header line of column names
    (fMRIPrep's ``*_desc-confounds_timeseries.tsv`` layout); ``columns`` selects and orders columns by name
    (default: every column), and ``n/a`` (or an empty field) is read as NaN -- harmless on a censored frame,
    rejected on a kept one.
    """
    ext = path.lower()
    if ext.endswith(".npy"):
        a = np.asarray(np.load(path), dtype=np.float64)
        if a.ndim == 1:
            a = a[:, None]
        if a.ndim != 2:
            raise ValueError("%s: expected a (T, K) array, got shape %s" % (path, a.shape))
        return np.ascontiguousarray(a if columns is None else a[:, list(columns)])
    if not ext.endswith((".tsv", ".csv")):
        raise ValueError("unsupported confounds file: %s" % path)
    delim = "\t" if ext.endswith(".tsv") else ","
    with open(path) as f:
        lines = [ln.rstrip("\r\n") for ln in f if ln.strip()]
    if not lines:
        raise ValueError("%s: empty confounds table" % path)
    names = [h.strip().strip('"') for h in lines[0].split(delim)]
    idx = list(range(len(names)))
    if columns is not None:
        missing = [c for c in columns if c not in names]
        if missing:
            raise ValueError("%s: no column(s) %s" % (path, missing))
        idx = [names.index(c) for c in columns]

    def value(tok):
        tok = tok.strip().strip('"')
        return np.nan if tok.lower() in ("n/a", "nan", "") else float(tok)

    rows = []
    for (i, ln) in enumerate(lines[1:], start=2):
        toks = ln.split(delim)
        if len(toks) != len(names):
            raise ValueError("%s:%d: %d fields, the header has %d" % (path, i, len(toks), len(names)))
        rows.append([value(toks[j]) for j in idx])
    return np.array(rows, dtype=np.float64).reshape(len(rows), len(idx))


def cleaned_correlations_from_files(control_paths, patient_paths, confound_paths=None, confound_columns=None,
                                    sample_masks=None, fisher=True, missing=False, time_major=False,
                                    kind="pearson", shrinkage="ledoit-wolf"):
    """(b, bt) as ``correlations_from_files`` returns them, from cleaned time series: subjects may differ in
    length; ``sample_masks`` (one (T_s,) bool array per subject, controls then patients) censors frames;
    ``confound_paths`` (one file per subject, same order) with ``confound_columns`` gives the regressors
    projected out of every region (``corr.correlations``); ``kind`` / ``shrinkage`` as there."""
    paths = list(control_paths) + list(patient_paths)
    ts = load_timeseries_list(paths, time_major)
    conf = None
    if confound_paths is not None:
        confound_paths = list(confound_paths)
        if len(confound_paths) != len(paths):
            raise ValueError("%d confound files for %d subjects" % (len(confound_paths), len(paths)))
        conf = [load_confounds(p, confound_columns) for p in confound_paths]
    masks = None if sample_masks is None else [np.asarray(m, dtype=bool) for m in sample_masks]
    c = corr.correlations(ts, fisher=fisher, missing=missing, sample_mask=masks, confounds=conf, kind=kind,
                          shrinkage=shrinkage)
    H = len(control_paths)
    return np.ascontiguousarray(c[:, :H]), np.ascontiguousarray(c[:, H:])
