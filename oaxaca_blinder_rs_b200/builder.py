"""Python mirror of the reference's builder / pyo3 surface for the bootstrap path, over the C ABI in
include/obboot_builder.h (the builder logic itself is the C++ host layer, csrc/host/builder.cc).

  OaxacaBuilder        builder.rs:37-246, :711-757, :787-951   (same method names)
  ReferenceCoefficients decomposition.rs:5-20
  OaxacaResults / TwoFoldResults / DecompositionDetail / ComponentResult   types.rs:10-47, :162-180
  OaxacaBlinder        python.rs:193-256 (fit / fit_quantile; module currently compiled out upstream)
  QuantileDecompositionBuilder / QuantileDecompositionResults / QuantileDecompositionDetail (Machado-Mata)
                       quantile_decomposition.rs:21-100, :281-421, :425-522

Frames are dicts of columns, pandas DataFrames or pyarrow Tables (polars is not in this image): float columns
become f64 columns (NaN/None = null), everything else string columns (None = null).
"""
from __future__ import annotations

import ctypes as C
import enum
import json
from types import SimpleNamespace
from typing import Iterable, List, Optional, Sequence

import numpy as np

from . import _native as N
from .core import OaxacaError


class ReferenceCoefficients(enum.IntEnum):
    GroupA = 0
    GroupB = 1
    Pooled = 2
    Weighted = 3
    Cotton = 4
    Neumark = 5


_bl = None


def _blib():
    global _bl
    if _bl is None:
        L = N.lib()
        vp, cp, i32, i64 = C.c_void_p, C.c_char_p, C.c_int32, C.c_int64
        L.ob_frame_new.restype = vp
        L.ob_frame_free.argtypes = [vp]; L.ob_frame_free.restype = None
        L.ob_frame_add_f64.argtypes = [vp, cp, N._DP, C.POINTER(C.c_uint8), i64]
        L.ob_frame_add_str.argtypes = [vp, cp, C.POINTER(cp), i64]
        L.ob_frame_read_csv.argtypes = [cp, C.POINTER(vp), C.c_char_p, C.c_size_t]
        L.ob_builder_new.argtypes = [vp, cp, cp, cp]; L.ob_builder_new.restype = vp
        L.ob_builder_from_formula.argtypes = [vp, cp, cp, cp, C.POINTER(vp), C.c_char_p, C.c_size_t]
        L.ob_builder_free.argtypes = [vp]; L.ob_builder_free.restype = None
        for fn in ("predictors", "categorical_predictors", "normalize"):
            getattr(L, "ob_builder_" + fn).argtypes = [vp, C.POINTER(cp), i32]
        L.ob_builder_weights.argtypes = [vp, cp]
        L.ob_builder_bootstrap_reps.argtypes = [vp, i64]
        L.ob_builder_reference_coefficients.argtypes = [vp, i32]
        L.ob_builder_heckman_selection.argtypes = [vp, cp, C.POINTER(cp), i32]
        L.ob_builder_cluster.argtypes = [vp, cp, i32]
        L.ob_builder_bayesian.argtypes = [vp, i32]
        L.ob_builder_seed.argtypes = [vp, C.c_uint64]
        L.ob_builder_device.argtypes = [vp, i32]
        L.ob_builder_index_stream.argtypes = [vp, N._U32P, N._U32P]
        L.ob_builder_run.argtypes = [vp, C.POINTER(vp)]
        L.ob_builder_run_outcomes.argtypes = [vp, C.POINTER(cp), i32, C.POINTER(vp)]
        L.ob_builder_decompose_quantile.argtypes = [vp, C.c_double, C.POINTER(vp)]
        L.ob_builder_get_data_matrices.argtypes = [vp, C.POINTER(i64), C.POINTER(i64), C.POINTER(i32), N._DP, N._DP, N._DP, N._DP]
        L.ob_builder_last_error.argtypes = [vp]; L.ob_builder_last_error.restype = cp
        L.ob_builder_describe.argtypes = [vp]; L.ob_builder_describe.restype = cp
        L.ob_builder_last_status.argtypes = [vp]
        L.ob_results_free.argtypes = [vp]; L.ob_results_free.restype = None
        L.ob_results_json.argtypes = [vp, i32, i32]; L.ob_results_json.restype = cp
        L.ob_results_summary.argtypes = [vp]; L.ob_results_summary.restype = cp
        L.ob_results_markdown.argtypes = [vp]; L.ob_results_markdown.restype = cp
        L.ob_results_residuals.argtypes = [vp, N._DP]; L.ob_results_residuals.restype = i64
        L.ob_qd_builder_new.argtypes = [vp, cp, cp, cp]; L.ob_qd_builder_new.restype = vp
        L.ob_qd_builder_free.argtypes = [vp]; L.ob_qd_builder_free.restype = None
        for fn in ("predictors", "categorical_predictors"):
            getattr(L, "ob_qd_builder_" + fn).argtypes = [vp, C.POINTER(cp), i32]
        L.ob_qd_builder_quantiles.argtypes = [vp, N._DP, i32]
        L.ob_qd_builder_simulations.argtypes = [vp, i64]
        L.ob_qd_builder_bootstrap_reps.argtypes = [vp, i64]
        L.ob_qd_builder_seed.argtypes = [vp, C.c_uint64]
        L.ob_qd_builder_device.argtypes = [vp, i32]
        L.ob_qd_builder_streams.argtypes = [vp, N._U32P, N._U32P, N._DP, N._U32P, N._U32P]
        L.ob_qd_builder_run.argtypes = [vp, C.POINTER(vp)]
        L.ob_qd_builder_last_error.argtypes = [vp]; L.ob_qd_builder_last_error.restype = cp
        L.ob_qd_builder_last_status.argtypes = [vp]
        L.ob_qd_quantile_key.argtypes = [C.c_double, C.c_char_p, C.c_size_t]; L.ob_qd_quantile_key.restype = i32
        L.ob_qd_results_free.argtypes = [vp]; L.ob_qd_results_free.restype = None
        L.ob_qd_results_json.argtypes = [vp]; L.ob_qd_results_json.restype = cp
        L.ob_qd_results_summary.argtypes = [vp]; L.ob_qd_results_summary.restype = cp
        _bl = L
    return _bl


BUILDER_SYMBOLS = ["ob_frame_new", "ob_frame_free", "ob_frame_add_f64", "ob_frame_add_str", "ob_frame_read_csv",
                   "ob_builder_new", "ob_builder_from_formula", "ob_builder_free", "ob_builder_predictors",
                   "ob_builder_categorical_predictors", "ob_builder_normalize", "ob_builder_weights",
                   "ob_builder_bootstrap_reps", "ob_builder_reference_coefficients", "ob_builder_heckman_selection",
                   "ob_builder_cluster", "ob_builder_bayesian", "ob_builder_seed", "ob_builder_device", "ob_builder_index_stream", "ob_builder_run", "ob_builder_run_outcomes",
                   "ob_builder_decompose_quantile", "ob_builder_get_data_matrices", "ob_builder_describe", "ob_builder_last_error", "ob_builder_last_status",
                   "ob_results_free", "ob_results_json", "ob_results_summary", "ob_results_markdown",
                   "ob_results_residuals",
                   "ob_qd_builder_new", "ob_qd_builder_free", "ob_qd_builder_predictors", "ob_qd_builder_categorical_predictors",
                   "ob_qd_builder_quantiles", "ob_qd_builder_simulations", "ob_qd_builder_bootstrap_reps", "ob_qd_builder_seed",
                   "ob_qd_builder_device", "ob_qd_builder_streams", "ob_qd_builder_run", "ob_qd_builder_last_error",
                   "ob_qd_builder_last_status", "ob_qd_quantile_key", "ob_qd_results_free", "ob_qd_results_json", "ob_qd_results_summary"]


def _columns(frame) -> dict:
    if isinstance(frame, dict):
        return frame
    if hasattr(frame, "to_pydict"):                      # pyarrow.Table
        return frame.to_pydict()
    if hasattr(frame, "columns") and hasattr(frame, "__getitem__"):   # pandas.DataFrame
        out = {}
        for c in frame.columns:
            col = frame[c]
            kind = getattr(getattr(col, "dtype", None), "kind", "O")
            # numeric columns stay numpy arrays (NaN = null): no per-value Python objects for large frames
            if kind in "fiu":
                try:
                    out[str(c)] = col.to_numpy(dtype=np.float64, na_value=np.nan)     # nullable Int64 / Float64 included
                except TypeError:
                    out[str(c)] = col.to_numpy(dtype=np.float64)
                continue
            # missing values as pandas itself sees them: None, NaN, pd.NA ('string' / nullable dtypes), NaT -- the
            # reference drops such rows (clean_dataframe, builder.rs:760-784); str(pd.NA) must never become a level
            mask = np.asarray(col.isna()) if hasattr(col, "isna") else None
            vals = col.tolist()
            out[str(c)] = [None if ((mask is not None and mask[i]) or v is None or (isinstance(v, float) and v != v)) else v
                           for i, v in enumerate(vals)]
        return out
    raise TypeError("dataframe must be a dict of columns, a pandas DataFrame or a pyarrow Table")


class _Frame:
    def __init__(self, frame):
        L = _blib()
        if isinstance(frame, _Frame):                    # e.g. read_csv(): share the native frame
            self._h, self._owner = frame._h, frame
            return
        self._owner = None
        self._h = C.c_void_p(L.ob_frame_new())
        for name, col in _columns(frame).items():
            vals = list(col) if not isinstance(col, np.ndarray) else col
            is_num = isinstance(vals, np.ndarray) and vals.dtype.kind in "fiu" or (
                not isinstance(vals, np.ndarray) and all(v is None or isinstance(v, (int, float, np.floating, np.integer))
                                                         for v in vals) and any(v is not None for v in vals))
            n = len(vals)
            if is_num:
                arr = np.array([np.nan if v is None else v for v in vals], dtype=np.float64) \
                    if not isinstance(vals, np.ndarray) else vals.astype(np.float64)
                valid = (~np.isnan(arr)).astype(np.uint8)
                vp = None if valid.all() else valid.ctypes.data_as(C.POINTER(C.c_uint8))
                arr = np.ascontiguousarray(np.nan_to_num(arr))
                st = L.ob_frame_add_f64(self._h, name.encode(), arr.ctypes.data_as(N._DP), vp, n)
            else:
                enc = (C.c_char_p * max(n, 1))(*[None if v is None else str(v).encode() for v in vals])
                st = L.ob_frame_add_str(self._h, name.encode(), enc, n)
            if st != 0:
                raise OaxacaError(st, f"Polars error: column {name}")

    def __del__(self):
        try:
            if self._h and self._owner is None:
                _blib().ob_frame_free(self._h)
        except Exception:
            pass


def read_csv(path: str) -> _Frame:
    """LazyCsvReader::new(path).with_has_header(true) (main.rs:161-165) through the native reader: a column is f64 if
    every non-empty cell parses as a number, empty cells are nulls.  Pass the result as `dataframe`."""
    L = _blib()
    f = _Frame.__new__(_Frame)
    f._owner = None
    h, err = C.c_void_p(), C.create_string_buffer(512)
    st = L.ob_frame_read_csv(str(path).encode(), C.byref(h), err, 512)
    if st != 0:
        raise OaxacaError(st, err.value.decode())
    f._h = h
    return f


def _names(names: Iterable[str]):
    v = [str(s).encode() for s in names]
    return (C.c_char_p * max(len(v), 1))(*v), len(v)


class ComponentResult(SimpleNamespace):
    """types.rs:172-180: name, estimate, std_err, t_stat, p_value, ci_lower, ci_upper."""


def _comps(rows):
    return [ComponentResult(**{k: (float("nan") if v is None else v) for k, v in r.items()}) for r in rows]


class OaxacaResults:
    """types.rs:24-47 (+ residuals / xa_mean / xb_mean / beta_star, the #[serde(skip)] fields)."""

    def __init__(self, handle):
        L = _blib()
        self._h = handle
        d = json.loads(L.ob_results_json(handle, 0, 1).decode())
        self.total_gap = d["total_gap"]
        tf = d["two_fold"]
        self.two_fold = SimpleNamespace(aggregate=_comps(tf["aggregate"]), detailed_explained=_comps(tf["detailed_explained"]),
                                        detailed_unexplained=_comps(tf["detailed_unexplained"]),
                                        detailed_selection=_comps(tf["detailed_selection"]))
        self.three_fold = SimpleNamespace(aggregate=_comps(d["three_fold"]["aggregate"]), detailed=_comps(d["three_fold"]["detailed"]))
        self.n_a, self.n_b = d["n_a"], d["n_b"]
        self.xa_mean, self.xb_mean = np.array(d["xa_mean"]), np.array(d["xb_mean"])
        self.beta_star = np.array(d["beta_star"])
        self.bootstrap_reps, self.successful_bootstraps = d["bootstrap_reps"], d["successful_bootstraps"]
        self.predictor_names = d["predictor_names"]
        self.timings_ms = dict(total=d["ms_total"], gram=d["ms_gram"])
        self.clusters = d.get("clusters")        # dict(strata, units_a, units_b) on a cluster bootstrap, else None
        self.bootstrap_scheme = d.get("bootstrap_scheme", "multinomial")
        n = L.ob_results_residuals(handle, None)
        self.residuals = np.empty(n)
        L.ob_results_residuals(handle, self.residuals.ctypes.data_as(N._DP))

    def explained(self):
        return next(c for c in self.two_fold.aggregate if c.name == "explained")      # types.rs:50-55

    def unexplained(self):
        return next(c for c in self.two_fold.aggregate if c.name == "unexplained")

    def summary(self) -> str:
        s = _blib().ob_results_summary(self._h).decode()
        print(s, end="")
        return s

    def to_json(self) -> str:
        return _blib().ob_results_json(self._h, 1, 0).decode()

    def to_markdown(self) -> str:
        return _blib().ob_results_markdown(self._h).decode()

    def __del__(self):
        try:
            if self._h:
                _blib().ob_results_free(self._h)
        except Exception:
            pass


class OaxacaBuilder:
    """builder.rs: OaxacaBuilder::new(df, outcome, group, reference_group) and its setters."""

    def __init__(self, dataframe, outcome: str, group: str, reference_group: str, _formula: Optional[str] = None):
        L = _blib()
        self._frame = _Frame(dataframe)
        self._keep = []
        if _formula is None:
            self._h = C.c_void_p(L.ob_builder_new(self._frame._h, outcome.encode(), group.encode(), reference_group.encode()))
        else:
            h, err = C.c_void_p(), C.create_string_buffer(512)
            st = L.ob_builder_from_formula(self._frame._h, _formula.encode(), group.encode(), reference_group.encode(),
                                           C.byref(h), err, 512)
            if st != 0:
                raise OaxacaError(st, err.value.decode())
            self._h = h

    @classmethod
    def from_formula(cls, dataframe, formula: str, group: str, reference_group: str) -> "OaxacaBuilder":
        return cls(dataframe, "", group, reference_group, _formula=formula)     # builder.rs:139-160

    def _check(self, st):
        if st != 0:
            raise OaxacaError(st, _blib().ob_builder_last_error(self._h).decode())
        return self

    def predictors(self, predictors: Sequence[str]):
        a, n = _names(predictors)
        return self._check(_blib().ob_builder_predictors(self._h, a, n))

    def categorical_predictors(self, predictors: Sequence[str]):
        a, n = _names(predictors)
        return self._check(_blib().ob_builder_categorical_predictors(self._h, a, n))

    def normalize(self, vars: Sequence[str]):
        a, n = _names(vars)
        return self._check(_blib().ob_builder_normalize(self._h, a, n))

    def weights(self, weights: str):
        return self._check(_blib().ob_builder_weights(self._h, weights.encode()))

    def bootstrap_reps(self, reps: int):
        return self._check(_blib().ob_builder_bootstrap_reps(self._h, int(reps)))

    def reference_coefficients(self, reference: ReferenceCoefficients):
        return self._check(_blib().ob_builder_reference_coefficients(self._h, int(reference)))

    def heckman_selection(self, outcome: str, predictors: Sequence[str]):
        a, n = _names(predictors)
        return self._check(_blib().ob_builder_heckman_selection(self._h, outcome.encode(), a, n))

    def seed(self, seed: int):
        return self._check(_blib().ob_builder_seed(self._h, int(seed)))

    def cluster(self, column: Optional[str], strata: Optional[str] = "group"):
        """Cluster bootstrap: resample whole clusters of `column` (string or numeric labels) instead of rows.  strata
        "group": a unit is a (cluster, group) pair and each group resamples its own units; "joint": one stratum, a drawn
        cluster brings its rows of both groups; None: resample rows again.  The column joins the null filter."""
        from .core import CLUSTER_NONE, CLUSTER_STRATA
        if strata is None or column is None:
            return self._check(_blib().ob_builder_cluster(self._h, None, CLUSTER_NONE))
        if strata not in CLUSTER_STRATA:
            raise ValueError(f"strata must be 'group', 'joint' or None, not {strata!r}")
        return self._check(_blib().ob_builder_cluster(self._h, column.encode(), CLUSTER_STRATA[strata]))

    def bayesian_bootstrap(self, on: bool = True):
        """Bayesian bootstrap: every row keeps a Dirichlet weight n_g E_i / sum E (E ~ Exp(1)) in every replicate instead of
        a multinomial count, so no replicate loses a rare categorical level.  run, run_outcomes and decompose_quantile
        honour it."""
        return self._check(_blib().ob_builder_bayesian(self._h, int(bool(on))))

    def device(self, device: int):
        return self._check(_blib().ob_builder_device(self._h, int(device)))

    def index_stream(self, idx_a, idx_b):
        """Test-only explicit resample index stream [reps x n_a], [reps x n_b] (row positions within each group).  Under
        cluster(): unit positions, [reps x units_a], [reps x units_b], or idx_a [reps x M] and idx_b=None for joint strata."""
        ia = np.ascontiguousarray(idx_a, dtype=np.uint32)
        ib = None if idx_b is None else np.ascontiguousarray(idx_b, dtype=np.uint32)
        self._keep = [ia, ib]
        return self._check(_blib().ob_builder_index_stream(self._h, ia.ctypes.data_as(N._U32P),
                                                           None if ib is None else ib.ctypes.data_as(N._U32P)))

    def run(self) -> OaxacaResults:                                  # builder.rs:787
        out = C.c_void_p()
        self._check(_blib().ob_builder_run(self._h, C.byref(out)))
        return OaxacaResults(out)

    def run_outcomes(self, outcomes) -> List["OaxacaResults"]:
        """run() once per listed outcome column on one ingest of the frame: rows are cleaned over every listed column, the
        first run fills a per-replicate Gram cache and the others contract only their outcome columns.  When the columns
        share their nulls, result k equals run() with outcomes[k] as the outcome."""
        names = [str(o) for o in outcomes]
        arr = (C.c_char_p * max(len(names), 1))(*[o.encode() for o in names])
        outs = (C.c_void_p * max(len(names), 1))()
        self._check(_blib().ob_builder_run_outcomes(self._h, arr, len(names), outs))
        return [OaxacaResults(C.c_void_p(outs[k])) for k in range(len(names))]

    def decompose_quantile(self, quantile: float) -> OaxacaResults:  # builder.rs:711
        out = C.c_void_p()
        self._check(_blib().ob_builder_decompose_quantile(self._h, float(quantile), C.byref(out)))
        return OaxacaResults(out)

    def describe(self) -> dict:
        """Host-only view of the cleaned / coded frame (no device needed): names, base names, n_a, n_b, normalize spec."""
        s = _blib().ob_builder_describe(self._h).decode()
        if not s:
            raise OaxacaError(_blib().ob_builder_last_status(self._h), _blib().ob_builder_last_error(self._h).decode())
        return json.loads(s)

    def get_data_matrices(self):                                     # builder.rs:252: (X_A, y_A, X_B, y_B)
        L = _blib()
        na, nb, k = C.c_int64(), C.c_int64(), C.c_int32()
        self._check(L.ob_builder_get_data_matrices(self._h, C.byref(na), C.byref(nb), C.byref(k), None, None, None, None))
        xa, ya = np.empty((na.value, k.value)), np.empty(na.value)
        xb, yb = np.empty((nb.value, k.value)), np.empty(nb.value)
        self._check(L.ob_builder_get_data_matrices(self._h, None, None, None, xa.ctypes.data_as(N._DP), ya.ctypes.data_as(N._DP),
                                                   xb.ctypes.data_as(N._DP), yb.ctypes.data_as(N._DP)))
        return xa, ya, xb, yb

    def __del__(self):
        try:
            if self._h:
                _blib().ob_builder_free(self._h)
        except Exception:
            pass


class OaxacaBlinder:
    """pyo3 surface (python.rs:193-256): OaxacaBlinder(dataframe, outcome, group, reference_group, predictors,
    categorical_predictors=[], bootstrap_reps=100, weights=None, ...).fit() / .fit_quantile(q)."""

    def __init__(self, dataframe, outcome, group, reference_group, predictors, categorical_predictors=(),
                 bootstrap_reps=100, weights=None, selection_outcome=None, selection_predictors=None):
        self._b = OaxacaBuilder(dataframe, outcome, group, reference_group)
        self._b.predictors(list(predictors)).categorical_predictors(list(categorical_predictors)).bootstrap_reps(bootstrap_reps)
        if weights is not None:
            self._b.weights(weights)
        if selection_outcome is not None:
            self._b.heckman_selection(selection_outcome, list(selection_predictors or []))

    def fit(self) -> OaxacaResults:
        try:
            return self._b.run()
        except OaxacaError as e:                      # python.rs:244: PyRuntimeError(str)
            raise RuntimeError(str(e)) from e

    def fit_quantile(self, quantile: float) -> OaxacaResults:
        try:
            return self._b.decompose_quantile(quantile)
        except OaxacaError as e:
            raise RuntimeError(str(e)) from e


class QuantileDecompositionDetail(SimpleNamespace):
    """quantile_decomposition.rs:512-522: total_gap, characteristics_effect, coefficients_effect (ComponentResult each)."""


class QuantileDecompositionResults:
    """quantile_decomposition.rs:425-437: results_by_quantile {"q25": detail, ..}, n_a, n_b (+ GPU-path bookkeeping)."""

    def __init__(self, handle):
        L = _blib()
        self._h = handle
        d = json.loads(L.ob_qd_results_json(handle).decode())
        self.results_by_quantile = {
            k: QuantileDecompositionDetail(**{name: _comps([v[name]])[0] for name in ("total_gap", "characteristics_effect", "coefficients_effect")})
            for k, v in d["results_by_quantile"].items()}
        self.n_a, self.n_b = d["n_a"], d["n_b"]
        self.bootstrap_reps, self.successful_bootstraps = d["bootstrap_reps"], d["successful_bootstraps"]
        self.qr = d["qr"]
        self.timings_ms = dict(total=d["ms_total"])

    def summary(self) -> str:
        s = _blib().ob_qd_results_summary(self._h).decode()
        print(s, end="")
        return s

    def to_json(self) -> str:
        return _blib().ob_qd_results_json(self._h).decode()

    def __del__(self):
        try:
            if self._h:
                _blib().ob_qd_results_free(self._h)
        except Exception:
            pass


class QuantileDecompositionBuilder:
    """quantile_decomposition.rs:21-100: QuantileDecompositionBuilder::new(df, outcome, group, reference_group) and its
    setters; defaults quantiles [0.1, 0.25, 0.5, 0.75, 0.9], 200 simulations, 20 bootstrap replications."""

    def __init__(self, dataframe, outcome: str, group: str, reference_group: str):
        L = _blib()
        self._frame = _Frame(dataframe)
        self._keep = []
        self._h = C.c_void_p(L.ob_qd_builder_new(self._frame._h, outcome.encode(), group.encode(), reference_group.encode()))

    def _check(self, st):
        if st != 0:
            raise OaxacaError(st, _blib().ob_qd_builder_last_error(self._h).decode())
        return self

    def predictors(self, predictors: Sequence[str]):
        a, n = _names(predictors)
        return self._check(_blib().ob_qd_builder_predictors(self._h, a, n))

    def categorical_predictors(self, predictors: Sequence[str]):
        a, n = _names(predictors)
        return self._check(_blib().ob_qd_builder_categorical_predictors(self._h, a, n))

    def quantiles(self, quantiles: Sequence[float]):
        q = np.ascontiguousarray(quantiles, dtype=np.float64)
        return self._check(_blib().ob_qd_builder_quantiles(self._h, q.ctypes.data_as(N._DP), len(q)))

    def simulations(self, reps: int):
        return self._check(_blib().ob_qd_builder_simulations(self._h, int(reps)))

    def bootstrap_reps(self, reps: int):
        return self._check(_blib().ob_qd_builder_bootstrap_reps(self._h, int(reps)))

    def seed(self, seed: int):
        return self._check(_blib().ob_qd_builder_seed(self._h, int(seed)))

    def device(self, device: int):
        return self._check(_blib().ob_qd_builder_device(self._h, int(device)))

    def streams(self, idx_a=None, idx_b=None, taus=None, draw_a=None, draw_b=None):
        """Test-only explicit streams (ob_mm_opts): resample indices [reps x n_g], random quantiles and simulated-row
        positions [(reps + 1) x simulations]."""
        u32 = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.uint32)
        ia, ib, da, db = u32(idx_a), u32(idx_b), u32(draw_a), u32(draw_b)
        t = None if taus is None else np.ascontiguousarray(taus, dtype=np.float64)
        self._keep = [ia, ib, t, da, db]
        p32 = lambda a: None if a is None else a.ctypes.data_as(N._U32P)
        return self._check(_blib().ob_qd_builder_streams(self._h, p32(ia), p32(ib), None if t is None else t.ctypes.data_as(N._DP),
                                                         p32(da), p32(db)))

    @staticmethod
    def quantile_key(tau: float) -> str:
        """format!("q{}", (tau * 100.0) as u32), quantile_decomposition.rs:277."""
        buf = C.create_string_buffer(32)
        _blib().ob_qd_quantile_key(float(tau), buf, 32)
        return buf.value.decode()

    def run(self) -> QuantileDecompositionResults:                   # quantile_decomposition.rs:281
        out = C.c_void_p()
        self._check(_blib().ob_qd_builder_run(self._h, C.byref(out)))
        return QuantileDecompositionResults(out)

    def __del__(self):
        try:
            if self._h:
                _blib().ob_qd_builder_free(self._h)
        except Exception:
            pass
