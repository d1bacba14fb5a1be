"""Numeric layer over the C ABI: Context, Design (packed in HBM), bootstrap().

Mirrors what OaxacaBuilder::run() does after the group split (builder.rs:808-950); the name-level
builder (strings, dummies, formula) lives in builder.py.  Every number comes from libobboot's CUDA
kernels -- nothing here computes on the CPU.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

from . import _native as N

REF_GROUP_A, REF_GROUP_B, REF_POOLED, REF_WEIGHTED = 0, 1, 2, 3


class OaxacaError(RuntimeError):
    """OaxacaError (error.rs:6-40) + device errors; .kind is the variant name."""

    def __init__(self, code: int, msg: str):
        self.code = code
        self.kind = N.STATUS_NAMES.get(code, str(code))
        super().__init__(msg or self.kind)


def _dp(a):
    return None if a is None else a.ctypes.data_as(N._DP)


def _ip(a):
    return None if a is None else a.ctypes.data_as(N._IP)


class Context:
    """ob_ctx: one per calling thread / GPU."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        st = N.lib().ob_ctx_create(device, C.byref(self._h))
        if st != 0:
            raise OaxacaError(st, f"ob_ctx_create(device={device}) failed: {N.STATUS_NAMES.get(st)} "
                                  f"(a B200 / sm_100a device is required; there is no CPU fallback)")
        self.device = device
        self.comm_world, self.comm_rank = 1, 0      # set by init_nccl / init_local

    def check(self, st: int):
        if st != 0:
            raise OaxacaError(st, N.lib().ob_last_error(self._h).decode())

    # ---- communicators for row sharding (mode N) ----
    def init_nccl(self, rank: int, world: int, group=None):
        """ob_comm_init_nccl: rank 0 creates the ncclUniqueId, torch.distributed only carries its 128 bytes."""
        import torch.distributed as dist
        ident = (C.c_uint8 * 128)()
        if rank == 0:
            st = N.lib().ob_comm_unique_id(ident)
            if st != 0:
                raise OaxacaError(st, "ob_comm_unique_id failed (libnccl.so.2 not loadable)")
        box = [bytes(ident)]
        dist.broadcast_object_list(box, src=0, group=group)
        ident = (C.c_uint8 * 128).from_buffer_copy(box[0])
        self.check(N.lib().ob_comm_init_nccl(self._h, ident, rank, world))
        self.comm_world, self.comm_rank = world, rank

    def init_local(self, group: "LocalGroup", rank: int):
        """ob_comm_init_local: one of several contexts (threads) of this process."""
        self.check(N.lib().ob_comm_init_local(self._h, group._h, rank))
        self._local_group = group          # keep the group alive as long as the communicator
        self.comm_world, self.comm_rank = group.world, rank

    def comm_destroy(self):
        if self._h:
            N.lib().ob_comm_destroy(self._h)
        self.comm_world, self.comm_rank = 1, 0

    def close(self):
        if self._h:
            N.lib().ob_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class LocalGroup:
    """ob_local_group: rendezvous of `world` contexts inside one process (threads)."""

    def __init__(self, world: int):
        self._h = C.c_void_p()
        st = N.lib().ob_local_group_create(world, C.byref(self._h))
        if st != 0:
            raise OaxacaError(st, "ob_local_group_create: 1 <= world <= 64")
        self.world = world

    def __del__(self):
        try:
            if self._h:
                N.lib().ob_local_group_destroy(self._h)
                self._h = C.c_void_p()
        except Exception:
            pass


def row_shard_plan(n_group: int, world: int, rank: int):
    """ob_row_shard_plan: [begin, end) positions (within the group, frame order) of the rows `rank` holds."""
    b, e = C.c_int64(), C.c_int64()
    st = N.lib().ob_row_shard_plan(n_group, world, rank, C.byref(b), C.byref(e))
    if st != 0:
        raise OaxacaError(st, "ob_row_shard_plan: world must be a power of two <= 64, 0 <= rank < world")
    return b.value, e.value


CACHE_NONE, CACHE_FILLED, CACHE_OUTCOME_ONLY, CACHE_SOLVE_ONLY = 0, 1, 2, 3
CLUSTER_NONE, CLUSTER_BY_GROUP, CLUSTER_JOINT = 0, 1, 2
CLUSTER_STRATA = {"group": CLUSTER_BY_GROUP, "joint": CLUSTER_JOINT}
CACHE_USE_NAMES = {CACHE_NONE: "none", CACHE_FILLED: "filled", CACHE_OUTCOME_ONLY: "outcome_only", CACHE_SOLVE_ONLY: "solve_only"}


class GramCache:
    """ob_gram_cache: every replicate's X'WX (and the last outcome's X'Wy) of one bootstrap configuration, kept in HBM.
    Pass it to bootstrap(..., cache=) on the same design across outcome changes (update_outcome, apply_rif*): the results
    are those of an uncached call bit for bit, while only the outcome columns of the Gram are contracted again."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        self._h = C.c_void_p()
        ctx.check(N.lib().ob_gram_cache_create(ctx._h, C.byref(self._h)))

    def _query(self):
        use, nbytes = C.c_int32(), C.c_int64()
        N.lib().ob_gram_cache_last_use(self._h, C.byref(use), C.byref(nbytes))
        return use.value, nbytes.value

    @property
    def last_use(self) -> int:
        """What the last cached bootstrap did: CACHE_FILLED, CACHE_OUTCOME_ONLY, CACHE_SOLVE_ONLY (CACHE_NONE: no call yet,
        or the last one failed)."""
        return self._query()[0]

    @property
    def bytes(self) -> int:
        """Device memory the cache holds."""
        return self._query()[1]

    def debug_cells(self) -> dict:
        """ob_debug_gram_cache_read: the reduced Gram cells the last cached bootstrap left here.  xx [2, slots, K(K+1)/2]
        (X'WX upper triangle, row-major), yy [2, slots, K T + 1] ((j, y_t) j-major, then (y_0, y_0)), rows [2, slots] (group
        row counts of a clustered design, else None), slots, K, T, count_bytes.  Slot 0 is the point estimate."""
        shape = np.zeros(5, dtype=np.int64)
        I64P = C.POINTER(C.c_int64)
        self.ctx.check(N.lib().ob_debug_gram_cache_read(self.ctx._h, self._h, shape.ctypes.data_as(I64P), None, None, None))
        slots, K, T, cb, has_rows = (int(v) for v in shape)
        xx = np.empty((2, slots, K * (K + 1) // 2))
        yy = np.empty((2, slots, K * T + 1))
        rows = np.empty((2, slots), dtype=np.int64) if has_rows else None
        self.ctx.check(N.lib().ob_debug_gram_cache_read(self.ctx._h, self._h, None, _dp(xx), _dp(yy),
                                                        None if rows is None else rows.ctypes.data_as(I64P)))
        return dict(xx=xx, yy=yy, rows=rows, slots=slots, K=K, T=T, count_bytes=cb)

    def close(self):
        if self._h:
            N.lib().ob_gram_cache_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


@dataclass
class NormVar:
    m: int
    idx: Sequence[int]
    has_base: bool = True


class Design:
    """ob_design: both groups' packed design matrices resident in HBM."""

    def __init__(self, ctx: Context, handle: C.c_void_p):
        self.ctx, self._h = ctx, handle
        na, nb, K, nc = C.c_int64(), C.c_int64(), C.c_int32(), C.c_int32()
        N.lib().ob_design_shape(self._h, C.byref(na), C.byref(nb), C.byref(K), C.byref(nc))
        self.n_a, self.n_b, self.K, self.n_cont = na.value, nb.value, K.value, nc.value
        ga, gb, w, r = C.c_int64(), C.c_int64(), C.c_int32(), C.c_int32()
        N.lib().ob_design_row_shard(self._h, C.byref(ga), C.byref(gb), C.byref(w), C.byref(r))
        self.n_a_global, self.n_b_global, self.world, self.rank = ga.value, gb.value, w.value, r.value
        self._inflight = None          # host columns an asynchronous pack is still reading

    @classmethod
    def from_dense(cls, ctx: Context, Xa, ya, wa, Xb, yb, wb, n_cont: int) -> "Design":
        Xa = np.ascontiguousarray(Xa, dtype=np.float64)
        Xb = np.ascontiguousarray(Xb, dtype=np.float64)
        K = Xa.shape[1]
        ya = np.ascontiguousarray(ya, dtype=np.float64)
        yb = np.ascontiguousarray(yb, dtype=np.float64)
        wa = None if wa is None else np.ascontiguousarray(wa, dtype=np.float64)
        wb = None if wb is None else np.ascontiguousarray(wb, dtype=np.float64)
        h = C.c_void_p()
        ctx.check(N.lib().ob_design_from_dense(ctx._h, K, n_cont, _dp(Xa), _dp(ya), _dp(wa), Xa.shape[0],
                                               _dp(Xb), _dp(yb), _dp(wb), Xb.shape[0], C.byref(h)))
        return cls(ctx, h)

    @classmethod
    def pack(cls, ctx: Context, cont: Sequence[np.ndarray], cat_codes: Sequence[np.ndarray],
             cat_levels: Sequence[int], outcome, weights, group, asynchronous: bool = False,
             row_shard: bool = False) -> "Design":
        """ob_design_pack from host columns (the cleaned, coded frame at builder.rs:808).
        asynchronous=True: ob_design_pack_async -- returns once the group split is known; the columns (keep them alive
        and unmodified, ideally in page-locked memory) are uploaded and packed under the first kernels of the next
        bootstrap() call.  The design keeps references to the arrays until then."""
        outcome = np.ascontiguousarray(outcome, dtype=np.float64)
        n = outcome.shape[0]
        cont = [np.ascontiguousarray(c, dtype=np.float64) for c in cont]
        cats = [np.ascontiguousarray(c, dtype=np.int32) for c in cat_codes]
        group = np.ascontiguousarray(group, dtype=np.uint8)
        weights = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64)
        assert all(c.shape == (n,) for c in cont + cats) and group.shape == (n,)
        fv = N.FrameView()
        fv.n, fv.n_cont, fv.n_cat = n, len(cont), len(cats)
        cont_arr = (N._DP * max(len(cont), 1))(*[_dp(c) for c in cont])
        cat_arr = (N._IP * max(len(cats), 1))(*[_ip(c) for c in cats])
        lv = np.array(list(cat_levels) + [0], dtype=np.int32)
        fv.cont, fv.cat_codes, fv.cat_levels = cont_arr, cat_arr, _ip(lv)
        fv.outcome, fv.weights = _dp(outcome), _dp(weights)
        fv.group = group.ctypes.data_as(C.POINTER(C.c_uint8))
        h = C.c_void_p()
        if row_shard:
            # ob_design_pack_row_shard_async (collective): the columns are THIS RANK'S frame slice, the result its row shard
            ctx.check(N.lib().ob_design_pack_row_shard_async(ctx._h, C.byref(fv), C.byref(h)))
            des = cls(ctx, h)
            des._inflight = (cont, cats, outcome, weights, group)
            return des
        if asynchronous:
            ctx.check(N.lib().ob_design_pack_async(ctx._h, C.byref(fv), C.byref(h)))
            des = cls(ctx, h)
            des._inflight = (cont, cats, outcome, weights, group)     # the upload reads these until the first use / wait()
            return des
        ctx.check(N.lib().ob_design_pack(ctx._h, C.byref(fv), C.byref(h)))
        return cls(ctx, h)

    def wait(self):
        """ob_design_wait: completes an asynchronous pack (raises its deferred errors)."""
        self.ctx.check(N.lib().ob_design_wait(self.ctx._h, self._h))
        self._inflight = None

    def download(self):
        """get_data_matrices() equivalent (builder.rs:252-291): (Xa, ya, wa, Xb, yb, wb) row-major."""
        Xa, Xb = np.empty((self.n_a, self.K)), np.empty((self.n_b, self.K))
        ya, yb, wa, wb = np.empty(self.n_a), np.empty(self.n_b), np.full(self.n_a, np.nan), np.full(self.n_b, np.nan)
        self.ctx.check(N.lib().ob_design_download(self.ctx._h, self._h, _dp(Xa), _dp(ya), _dp(wa), _dp(Xb), _dp(yb), _dp(wb)))
        return Xa, ya, wa, Xb, yb, wb

    def allgather_rows(self) -> "Design":
        """ob_design_allgather_rows: this design holds rank's contiguous frame slice; returns the full design
        (identical on every rank) assembled over the context's communicator."""
        h = C.c_void_p()
        self.ctx.check(N.lib().ob_design_allgather_rows(self.ctx._h, self._h, C.byref(h)))
        return Design(self.ctx, h)

    def redistribute_rows(self) -> "Design":
        """ob_design_redistribute_rows: this design holds rank's contiguous frame slice; returns rank's ROW SHARD (mode N),
        the rows exchanged over the context's communicator."""
        h = C.c_void_p()
        self.ctx.check(N.lib().ob_design_redistribute_rows(self.ctx._h, self._h, C.byref(h)))
        return Design(self.ctx, h)

    def pack_timings(self):
        """(ms_h2d, ms_pack_kernels) of the ob_design_pack call that built this design."""
        a, b = C.c_double(), C.c_double()
        N.lib().ob_design_pack_timings(self._h, C.byref(a), C.byref(b))
        return a.value, b.value

    def set_row_shard(self, n_a_global: int, n_b_global: int, world: int, rank: int):
        """ob_design_set_row_shard: this design holds rank's rows (row_shard_plan) of a world-way row split."""
        st = N.lib().ob_design_set_row_shard(self._h, n_a_global, n_b_global, world, rank)
        if st != 0:
            raise OaxacaError(st, f"ob_design_set_row_shard: local rows ({self.n_a}, {self.n_b}) do not match the plan "
                                  f"for rank {rank} of {world}")
        self.n_a_global, self.n_b_global, self.world, self.rank = n_a_global, n_b_global, world, rank

    def update_outcome(self, y_frame):
        """ob_design_update_outcome: new outcome (one value per frame row), X / weights / group split stay resident."""
        y = np.ascontiguousarray(y_frame, dtype=np.float64)
        self.ctx.check(N.lib().ob_design_update_outcome(self.ctx._h, self._h, _dp(y), y.shape[0]))

    def apply_rif(self, tau: float):
        self.ctx.check(N.lib().ob_design_apply_rif(self.ctx._h, self._h, float(tau)))

    def apply_rif_multi(self, taus: Sequence[float]):
        """ob_design_apply_rif_multi: one RIF outcome column per quantile; the next bootstrap() contracts the Gram once
        for all of them and returns every per-outcome array with a leading quantile dimension."""
        t = np.ascontiguousarray(list(taus), dtype=np.float64)
        self.ctx.check(N.lib().ob_design_apply_rif_multi(self.ctx._h, self._h, _dp(t), len(t)))

    def attach_selection(self, selection_outcome, selection_predictors: Sequence[np.ndarray]):
        """ob_design_attach_selection (OaxacaBuilder::heckman_selection, builder.rs:236-246): the binary selection outcome
        and the selection predictors, one value per row of the frame this design was packed from.  bootstrap() then runs
        the Heckman two-step estimator per replicate; coefficient / mean vectors gain the IMR entry (last) and the
        statistics the detailed_selection rows."""
        s = np.ascontiguousarray(selection_outcome, dtype=np.float64)
        preds = [np.ascontiguousarray(p, dtype=np.float64) for p in selection_predictors]
        assert all(p.shape == s.shape for p in preds)
        sv = N.SelectionView()
        sv.n_pred = len(preds)
        arr = (N._DP * max(len(preds), 1))(*[_dp(p) for p in preds])
        sv.pred, sv.outcome = arr, _dp(s)
        self.ctx.check(N.lib().ob_design_attach_selection(self.ctx._h, self._h, C.byref(sv), s.shape[0]))

    def attach_clusters(self, codes, n_codes: Optional[int] = None, strata: Optional[str] = "group"):
        """ob_design_attach_clusters: resample whole clusters instead of rows.  codes: one integer code in [0, n_codes) per
        row of the frame this design was packed from (n_codes defaults to max + 1); strata "group" (a unit is a (cluster,
        group) pair, each group resamples its own units), "joint" (one stratum: a drawn cluster brings its rows of both
        groups) or None (detach: rows are resampled again).  Units are numbered by ascending code; an explicit index stream
        passed to bootstrap() then draws units (see `clusters`)."""
        if strata is None:
            self.ctx.check(N.lib().ob_design_attach_clusters(self.ctx._h, self._h, None, 0, 0, CLUSTER_NONE))
            return
        if strata not in CLUSTER_STRATA:
            raise ValueError(f"strata must be 'group', 'joint' or None, not {strata!r}")
        c = np.ascontiguousarray(codes, dtype=np.int32)
        if n_codes is None:
            n_codes = int(c.max()) + 1 if c.size else 1
        self.ctx.check(N.lib().ob_design_attach_clusters(self.ctx._h, self._h, _ip(c), c.shape[0], int(n_codes),
                                                         CLUSTER_STRATA[strata]))

    @property
    def clusters(self) -> Optional[dict]:
        """None when rows are resampled, else dict(strata="group" | "joint", units_a=M_A, units_b=M_B) (joint: both = M)."""
        st, ua, ub = C.c_int32(), C.c_int64(), C.c_int64()
        N.lib().ob_design_clusters(self._h, C.byref(st), C.byref(ua), C.byref(ub))
        if st.value == CLUSTER_NONE:
            return None
        return dict(strata="joint" if st.value == CLUSTER_JOINT else "group", units_a=ua.value, units_b=ub.value)

    @property
    def selection_cols(self) -> int:
        k1 = C.c_int32()
        N.lib().ob_design_selection_cols(self._h, C.byref(k1))
        return k1.value

    @property
    def n_outcomes(self) -> int:
        t = C.c_int32()
        N.lib().ob_design_num_outcomes(self._h, C.byref(t))
        return t.value

    def debug_counts(self, seed: int, rep: int, group: int) -> np.ndarray:
        n = self.n_a if group == 0 else self.n_b
        out = np.empty(n, dtype=np.uint16)
        self.ctx.check(N.lib().ob_debug_counts(self.ctx._h, self._h, seed, rep, group,
                                               out.ctypes.data_as(C.POINTER(C.c_uint16))))
        return out

    def debug_bayes_weights(self, seed: int, rep: int, group: int) -> np.ndarray:
        """ob_debug_bayes_weights: the native Bayesian-bootstrap weights E (fp32, unnormalised) of global replicate `rep`
        of `group`, in row order."""
        out = np.empty(self.n_a if group == 0 else self.n_b, dtype=np.float32)
        self.ctx.check(N.lib().ob_debug_bayes_weights(self.ctx._h, self._h, seed, rep, group,
                                                      out.ctypes.data_as(C.POINTER(C.c_float))))
        return out

    def debug_counts_from_indices(self, idx, group: int, count_bits: int = 8):
        """ob_debug_counts_from_indices: (counts [reps, n_local] uint16, flags) of an explicit index stream
        idx [reps, n_global] through the production histogram kernel."""
        idx = np.ascontiguousarray(idx, dtype=np.uint32)
        n_loc = self.n_a if group == 0 else self.n_b
        n_glob = self.n_a_global if group == 0 else self.n_b_global
        assert idx.ndim == 2 and idx.shape[1] == n_glob
        out = np.empty((idx.shape[0], n_loc), dtype=np.uint16)
        flags = C.c_int32(0)
        self.ctx.check(N.lib().ob_debug_counts_from_indices(self.ctx._h, self._h, group, idx.ctypes.data_as(N._U32P),
                                                            idx.shape[0], count_bits,
                                                            out.ctypes.data_as(C.POINTER(C.c_uint16)), C.byref(flags)))
        return out, flags.value

    def close(self):
        if self._h:
            N.lib().ob_design_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def ingest(ctx: Context, cont, cat, outcome, weights, group, reference_group: str):
    """Device-side cleaning + coding + pack of a raw frame (ob_ingest_begin / ob_ingest_finish; builder.rs:760-806,
    :61-102).  Numeric columns: float64 arrays (NaN = null) or (array, valid_bytes) pairs (NaN or valid == 0 = null).  String columns come
    dictionary-encoded as (codes int32 with < 0 = null, dictionary list of str) -- e.g. pandas
    `Categorical.codes / .categories`, pyarrow `DictionaryArray.indices / .dictionary`.
    Returns (Design, meta) with meta = dict(rows_kept, group_a, levels per categorical (sorted; [0] is the base))."""
    U8P = C.POINTER(C.c_uint8)
    keep = []          # keep numpy temporaries alive across the calls

    def f64(col):
        if isinstance(col, tuple):
            data, valid = col
            data = np.ascontiguousarray(data, dtype=np.float64)
            valid = None if valid is None else np.ascontiguousarray(valid, dtype=np.uint8)
        else:
            data = np.ascontiguousarray(col, dtype=np.float64)     # NaN = null, detected on the device (nan_is_null)
            valid = None
        keep.extend([data, valid])
        r = N.RawF64()
        r.data = _dp(data)
        r.valid = None if valid is None else valid.ctypes.data_as(U8P)
        return r, data.shape[0]

    def dct(col):
        codes, dictionary = col
        codes = np.ascontiguousarray(codes, dtype=np.int32)
        keep.append(codes)
        r = N.RawDict()
        r.codes, r.dict_size = _ip(codes), len(dictionary)
        return r, [str(s) for s in dictionary]

    fr = N.RawFrame()
    fr.nan_is_null = 1
    conts = [f64(c)[0] for c in cont]
    cats, dicts = zip(*[dct(c) for c in cat]) if cat else ((), ())
    fr.outcome, n = f64(outcome)
    fr.n, fr.n_cont, fr.n_cat = n, len(conts), len(cats)
    cont_arr = (N.RawF64 * max(len(conts), 1))(*conts)
    cat_arr = (N.RawDict * max(len(cats), 1))(*cats)
    fr.cont, fr.cat = cont_arr, cat_arr
    if weights is not None:
        fr.weights = f64(weights)[0]
    fr.group, gdict = dct(group)
    h = C.c_void_p()
    ctx.check(N.lib().ob_ingest_begin(ctx._h, C.byref(fr), C.byref(h)))
    try:
        kept = C.c_int64()
        N.lib().ob_ingest_rows_kept(h, C.byref(kept))

        def present(col, size):
            out = np.zeros(max(size, 1), dtype=np.uint8)
            N.lib().ob_ingest_presence(h, col, out.ctypes.data_as(U8P))
            return out[:size].astype(bool)
        # split_groups (builder.rs:61-102): sorted unique values of the cleaned frame; A = first one that is not the reference
        gp = present(-1, len(gdict))
        groups = sorted({gdict[i] for i in np.flatnonzero(gp)})
        if len(groups) < 2:
            raise OaxacaError(3, "Invalid group variable: Not enough groups for comparison")
        group_a = groups[0] if groups[0] != reference_group else groups[1]
        gmap = np.array([0 if s == group_a else (1 if s == reference_group else 2) for s in gdict] + [2], dtype=np.int32)
        # create_dummies_manual (builder.rs:380-418): levels sorted ascending, first = base
        levels, remaps = [], []
        for q, dq in enumerate(dicts):
            pq = present(q, len(dq))
            lv = sorted({dq[i] for i in np.flatnonzero(pq)})
            if not lv:
                raise OaxacaError(3, "Invalid group variable: Could not get reference category")
            code = {s: i for i, s in enumerate(lv)}
            remaps.append(np.array([code[s] if pq[i] else -1 for i, s in enumerate(dq)] + [-1], dtype=np.int32))
            levels.append(lv)
        remap_arr = (N._IP * max(len(remaps), 1))(*[_ip(r) for r in remaps])
        lvl = np.array([len(lv) for lv in levels] + [0], dtype=np.int32)
        dh = C.c_void_p()
        ctx.check(N.lib().ob_ingest_finish(ctx._h, h, _ip(gmap), remap_arr, _ip(lvl), C.byref(dh)))
    finally:
        N.lib().ob_ingest_destroy(h)
    return Design(ctx, dh), dict(rows_kept=int(kept.value), group_a=group_a, levels=levels)


class PinnedBuffer:
    """ob_host_alloc: page-locked host memory as a numpy array (.array); freed on close() / garbage collection."""

    def __init__(self, shape, dtype=np.float64):
        self._p = C.c_void_p()
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        st = N.lib().ob_host_alloc(max(nbytes, 1), C.byref(self._p))
        if st != 0:
            raise OaxacaError(st, "ob_host_alloc failed")
        buf = (C.c_uint8 * max(nbytes, 1)).from_address(self._p.value)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def close(self):
        if self._p:
            self.array = None
            N.lib().ob_host_free(self._p)
            self._p = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def pin_in_place(arrays):
    """ob_host_register on existing numpy arrays (what a Rust caller does with the Vecs it already holds): returns the
    list of registered arrays; pass it to unpin() when done.  Arrays that cannot be registered are left pageable."""
    done = []
    for a in arrays:
        if a is None or a.nbytes == 0:
            continue
        if N.lib().ob_host_register(a.ctypes.data_as(C.c_void_p), a.nbytes) == 0:
            done.append(a)
    return done


def unpin(arrays):
    for a in arrays:
        N.lib().ob_host_unregister(a.ctypes.data_as(C.c_void_p))


def replicate_shard(reps: int, world: int, rank: int):
    """ob_replicate_shard: [begin, end) of the global replicate ids rank computes under shard_replicates."""
    b, e = C.c_int64(), C.c_int64()
    st = N.lib().ob_replicate_shard(reps, world, rank, C.byref(b), C.byref(e))
    if st != 0:
        raise OaxacaError(st, "ob_replicate_shard: bad arguments")
    return b.value, e.value


def num_stats(K: int, norm: Sequence[NormVar]) -> int:
    return 5 + 2 * (K + sum(1 for v in norm if v.has_base))


def bootstrap(design: Design, reps: int, ref_kind: int = REF_GROUP_A, norm: Sequence[NormVar] = (),
              seed: int = 0, idx_a=None, idx_b=None, rep_begin: int = 0, rep_end: int = 0,
              skip_reduce: bool = False, count_bits: int = 0, max_workspace_bytes: int = 0,
              want_rep: bool = False, want_residuals: bool = True, residuals_out: Optional[np.ndarray] = None,
              shard_replicates: bool = False, cache: Optional[GramCache] = None, scheme: str = "multinomial",
              wt_a=None, wt_b=None) -> dict:
    """ob_bootstrap_run (ob_bootstrap_run_cached with a GramCache: same results, and `cache_use` in the dict).  Returns point estimates, per-statistic SE/p/CI/t and (optionally) replicate detail.
    scheme "bayes": the Bayesian bootstrap (ob_bootstrap_run_bayes): every row keeps a Dirichlet weight n_g E_i / sum E
    with E ~ Exp(1) in every replicate.  wt_a [reps x n_a] / wt_b [reps x n_b]: a test-only explicit stream of E (float32);
    None = the native stream.
    On a clustered design (Design.attach_clusters) idx_a / idx_b draw units: [reps x units_a] / [reps x units_b], or
    idx_a [reps x M] with idx_b=None under joint strata.
    residuals_out: optional preallocated float64 [n_b] buffer for OaxacaResults.residuals (reusing one across calls
    avoids first-touch page faults on a fresh 8 n_b byte array during the device-to-host copy; a page-locked one --
    pinned_empty() -- takes the DMA directly).
    shard_replicates: mode R inside the library -- the context carries a communicator (init_nccl / init_local), every
    rank makes this same call on the whole design and gets the identical, gathered result (rep_* cover all reps)."""
    ctx, K = design.ctx, design.K
    norm = list(norm)
    S = num_stats(K, norm)
    K1 = design.selection_cols
    if K1:                      # Heckman: K + 1 coefficients (IMR last), no Yun rows, K1 detailed_selection rows
        norm, K = [], K + 1
        S = 5 + 2 * K + K1
    o = N.BootOpts()
    o.ref_kind, o.n_norm = ref_kind, len(norm)
    m = np.array([v.m for v in norm] + [0], dtype=np.int32)
    off = np.zeros(len(norm) + 1, dtype=np.int32)
    for i, v in enumerate(norm):
        off[i + 1] = off[i] + len(v.idx)
    idx = np.array([j for v in norm for j in v.idx] + [0], dtype=np.int32)
    hb = np.array([int(v.has_base) for v in norm] + [0], dtype=np.int32)
    o.norm_m, o.norm_off, o.norm_idx, o.norm_has_base = _ip(m), _ip(off), _ip(idx), _ip(hb)
    o.reps, o.seed = reps, seed
    if scheme not in ("multinomial", "bayes"):
        raise ValueError(f"scheme must be 'multinomial' or 'bayes', not {scheme!r}")
    bo = None
    if scheme == "bayes":
        bo = N.BayesOpts()
        if wt_a is not None or wt_b is not None:
            wt_a = np.ascontiguousarray(wt_a, dtype=np.float32)
            wt_b = np.ascontiguousarray(wt_b, dtype=np.float32)
            assert wt_a.shape == (reps, design.n_a_global) and wt_b.shape == (reps, design.n_b_global)
            bo.wt_a, bo.wt_b = wt_a.ctypes.data_as(C.POINTER(C.c_float)), wt_b.ctypes.data_as(C.POINTER(C.c_float))
    elif wt_a is not None or wt_b is not None:
        raise ValueError("wt_a / wt_b are weight streams of scheme='bayes'")
    cl = design.clusters
    if idx_a is not None and cl is not None and cl["strata"] == "joint":
        # one unit stream over both groups
        assert idx_b is None, "a joint cluster design takes one unit stream (idx_b=None)"
        idx_a = np.ascontiguousarray(idx_a, dtype=np.uint32)
        assert idx_a.shape == (reps, cl["units_a"])
        o.idx_a = idx_a.ctypes.data_as(N._U32P)
    elif idx_a is not None:
        idx_a = np.ascontiguousarray(idx_a, dtype=np.uint32)
        idx_b = np.ascontiguousarray(idx_b, dtype=np.uint32)
        n_a, n_b = (cl["units_a"], cl["units_b"]) if cl is not None else (design.n_a_global, design.n_b_global)
        assert idx_a.shape == (reps, n_a) and idx_b.shape == (reps, n_b)
        o.idx_a, o.idx_b = idx_a.ctypes.data_as(N._U32P), idx_b.ctypes.data_as(N._U32P)
    o.rep_begin, o.rep_end = rep_begin, rep_end
    o.skip_reduce, o.count_bits, o.max_workspace_bytes = int(skip_reduce), count_bits, max_workspace_bytes
    o.shard_replicates = int(shard_replicates)
    nrep = (rep_end if rep_end > 0 else reps) - rep_begin     # shard_replicates: rep_* outputs cover all reps rows

    r = N.Result()
    T = design.n_outcomes                  # > 1 after apply_rif_multi: a leading quantile dimension on per-outcome arrays
    lead = (T,) if T > 1 else ()
    a = dict(point_stats=np.empty(lead + (S,)), xa_mean=np.empty(K), xb_mean=np.empty(K), beta_star=np.empty(lead + (K,)),
             beta_a=np.empty(lead + (K,)), beta_b=np.empty(lead + (K,)), std_err=np.full(lead + (S,), np.nan),
             p_value=np.full(lead + (S,), np.nan), ci_lower=np.full(lead + (S,), np.nan), ci_upper=np.full(lead + (S,), np.nan),
             t_stat=np.zeros(lead + (S,)), total_gap_multi=np.empty(T))
    if K1:
        a["sel_gamma_a"], a["sel_gamma_b"] = np.empty(K1), np.empty(K1)
    if want_residuals:
        if residuals_out is not None:
            assert residuals_out.dtype == np.float64 and residuals_out.shape == lead + (design.n_b,) and residuals_out.flags.c_contiguous
        a["residuals_b"] = residuals_out if residuals_out is not None else np.empty(lead + (design.n_b,))
    if want_rep or skip_reduce:
        a["rep_stats"] = np.empty((max(nrep, 1),) + lead + (S,))
        a["rep_status"] = np.zeros(max(nrep, 1), dtype=np.int32)
        a["rep_beta_a"] = np.empty((max(nrep, 1),) + lead + (K,))
        a["rep_beta_b"] = np.empty((max(nrep, 1),) + lead + (K,))
    for k, v in a.items():
        setattr(r, k, _ip(v) if v.dtype == np.int32 else _dp(v))
    try:
        if bo is not None:
            ctx.check(N.lib().ob_bootstrap_run_bayes(ctx._h, design._h, C.byref(o), C.byref(bo),
                                                     None if cache is None else cache._h, C.byref(r)))
        elif cache is None:
            ctx.check(N.lib().ob_bootstrap_run(ctx._h, design._h, C.byref(o), C.byref(r)))
        else:
            ctx.check(N.lib().ob_bootstrap_run_cached(ctx._h, design._h, C.byref(o), cache._h, C.byref(r)))
    finally:
        design._inflight = None        # an asynchronous pack has completed (or failed) by now
    out = dict(a)
    if cache is not None:
        out["cache_use"] = cache.last_use
    for k in ("rep_stats", "rep_status", "rep_beta_a", "rep_beta_b"):
        if k in out:
            out[k] = out[k][:nrep]
    ps = a["point_stats"]
    out.update(total_gap=r.total_gap, n_ok=int(r.n_ok), S=S, n_outcomes=T,
               two_fold=ps[..., :2].copy(), three_fold=ps[..., 2:5].copy(),
               timings_ms=dict(counts=r.ms_counts, gram=r.ms_gram, gram_main=r.ms_gram_kernel, solve=r.ms_solve,
                               reduce=r.ms_reduce, total=r.ms_total, comm=r.ms_comm),
               gpu_launches=int(r.gpu_launches))
    D = (S - 5 - K1) // 2
    out["det_expl"], out["det_unexpl"] = ps[..., 5:5 + D].copy(), ps[..., 5 + D:5 + 2 * D].copy()
    if K1:
        out["det_selection"] = ps[..., 5 + 2 * D:].copy()
    return out


QR_VERTEX, QR_APPROX, QR_FAILED = 0, 1, 2


def machado_mata(design: Design, quantiles: Sequence[float] = (0.1, 0.25, 0.5, 0.75, 0.9), simulations: int = 200,
                 reps: int = 20, seed: int = 0, idx_a=None, idx_b=None, taus=None, draw_a=None, draw_b=None,
                 rep_begin: int = 0, rep_end: int = 0, skip_reduce: bool = False, count_bits: int = 0,
                 max_workspace_bytes: int = 0, want_rep: bool = False, want_betas: bool = False,
                 shard_replicates: bool = False) -> dict:
    """ob_mm_run: the Machado-Mata quantile decomposition (QuantileDecompositionBuilder::run,
    quantile_decomposition.rs:281-421) on a packed design.  Statistics per target quantile: (gap, characteristics,
    coefficients).  Explicit streams (tests): idx_a / idx_b [reps x n_g]; taus, draw_a, draw_b [(reps + 1) x simulations]
    (row 0 = the point pass; draws are positions in the pass's resampled group frame)."""
    ctx, K = design.ctx, design.K
    q = np.ascontiguousarray(quantiles, dtype=np.float64)
    nq, S = len(q), 3 * len(q)
    o = N.MmOpts()
    o.simulations, o.n_quantiles, o.quantiles, o.reps, o.seed = simulations, nq, _dp(q), reps, seed
    keep = []
    if idx_a is not None:
        idx_a = np.ascontiguousarray(idx_a, dtype=np.uint32)
        idx_b = np.ascontiguousarray(idx_b, dtype=np.uint32)
        assert idx_a.shape == (reps, design.n_a_global) and idx_b.shape == (reps, design.n_b_global)
        o.idx_a, o.idx_b = idx_a.ctypes.data_as(N._U32P), idx_b.ctypes.data_as(N._U32P)
    if taus is not None:
        taus = np.ascontiguousarray(taus, dtype=np.float64)
        assert taus.shape == (reps + 1, simulations)
        o.taus = _dp(taus)
    if draw_a is not None:
        draw_a = np.ascontiguousarray(draw_a, dtype=np.uint32)
        draw_b = np.ascontiguousarray(draw_b, dtype=np.uint32)
        assert draw_a.shape == (reps + 1, simulations) and draw_b.shape == (reps + 1, simulations)
        o.draw_a, o.draw_b = draw_a.ctypes.data_as(N._U32P), draw_b.ctypes.data_as(N._U32P)
    keep += [idx_a, idx_b, taus, draw_a, draw_b]
    o.rep_begin, o.rep_end = rep_begin, rep_end
    o.skip_reduce, o.count_bits, o.max_workspace_bytes = int(skip_reduce), count_bits, max_workspace_bytes
    o.shard_replicates = int(shard_replicates)
    nrep = (rep_end if rep_end > 0 else reps) - rep_begin
    r = N.MmResult()
    a = dict(point_stats=np.empty(S), std_err=np.full(S, np.nan), p_value=np.full(S, np.nan), ci_lower=np.full(S, np.nan),
             ci_upper=np.full(S, np.nan), t_stat=np.zeros(S))
    if want_rep or skip_reduce:
        a["rep_stats"] = np.empty((max(nrep, 1), S))
        a["rep_status"] = np.zeros(max(nrep, 1), dtype=np.int32)
    if want_betas:
        a["point_betas_a"], a["point_betas_b"] = np.empty((simulations, K)), np.empty((simulations, K))
        a["point_qr_info_a"], a["point_qr_info_b"] = np.zeros(simulations, dtype=np.int32), np.zeros(simulations, dtype=np.int32)
    for k, v in a.items():
        setattr(r, k, _ip(v) if v.dtype == np.int32 else _dp(v))
    try:
        ctx.check(N.lib().ob_mm_run(ctx._h, design._h, C.byref(o), C.byref(r)))
    finally:
        design._inflight = None
    out = dict(a)
    for k in ("rep_stats", "rep_status"):
        if k in out:
            out[k] = out[k][:nrep]
    for k in ("point_stats", "std_err", "p_value", "ci_lower", "ci_upper", "t_stat"):
        out[k] = out[k].reshape(nq, 3)
    if "rep_stats" in out:
        out["rep_stats"] = out["rep_stats"].reshape(-1, nq, 3)
    out.update(n_ok=int(r.n_ok), S=S, quantiles=q,
               qr=dict(total=int(r.qr_total), vertex=int(r.qr_vertex), approx=int(r.qr_approx), failed=int(r.qr_failed),
                       iterations=int(r.qr_iterations)),
               timings_ms=dict(counts=r.ms_counts, qr=r.ms_qr, effects=r.ms_effects, reduce=r.ms_reduce, total=r.ms_total),
               gpu_launches=int(r.gpu_launches))
    return out


def reduce_stats(ctx: Context, rep_stats, rep_status, point_stats) -> dict:
    """ob_reduce_stats on host arrays gathered from several shards (replicate order)."""
    rep_stats = np.ascontiguousarray(rep_stats, dtype=np.float64)
    reps, S = rep_stats.shape
    rep_status = np.ascontiguousarray(rep_status, dtype=np.int32)
    point_stats = np.ascontiguousarray(point_stats, dtype=np.float64)
    out = {k: np.empty(S) for k in ("std_err", "p_value", "ci_lower", "ci_upper", "t_stat")}
    nok = C.c_int64()
    ctx.check(N.lib().ob_reduce_stats(ctx._h, _dp(rep_stats), _ip(rep_status), reps, S, _dp(point_stats),
                                      C.byref(nok), *[_dp(out[k]) for k in
                                                      ("std_err", "p_value", "ci_lower", "ci_upper", "t_stat")]))
    out["n_ok"] = int(nok.value)
    return out
