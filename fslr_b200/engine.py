"""Host side of the B200 clustering step: owns buffers through PyTorch, calls the C ABI.

`Engine.cluster(table, params)` is the fused entry the benchmark and the drop-in functions of
fslr_b200.cluster use (SURVEY.md §8b `cluster_table`).  Threshold tables that depend on floating point
(`umax`, `1 - qlen_diff`, `1 - n_alignment_diff`) are computed here with Python floats — the reference's own
arithmetic (cluster.py:170,179,181,218-219) — so the device only ever compares integers.
"""
import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import _native
from .table import ClusterParams, ColumnarTable

_COLS = ("read_id", "chrom", "rstart", "rend", "aln_size", "qstart", "qend", "n_alignments")


def umax_table(cutoffs, n_max=_native.MAX_FILLINGS):
    """umax[n] = largest union u >= n with n/u >= cutoff(n) in float64; n-1 when none (cluster.py:165-170,218-219)."""
    out = [0]
    for n in range(1, n_max + 1):
        t = cutoffs[n - 1] if n - 1 < len(cutoffs) else cutoffs[-1]
        if t <= 0:
            out.append(2**31 - 1)
            continue
        u = min(int(n / t) + 2, 2**31 - 1)
        while u >= n and not (n / u >= t):
            u -= 1
        out.append(u if u >= n else n - 1)
    return out


@dataclass
class EdgeList:
    """The similarity graph of one clustering call (cluster.py:187-227's match_df / G), one row per edge handed to
    union-find: read1 is the read whose query tested the pair (match_df's query1), jaccard its Jaccard similarity in that
    direction.  Rows sorted by (query rank of read1, query rank of read2)."""
    read1: np.ndarray          # int32 read id
    read2: np.ndarray          # int32 read id
    jaccard: np.ndarray        # float64


@dataclass
class ClusterResult:
    cluster: np.ndarray        # int32 per read id: the `cluster` value main.py:334-342 writes for that read's rows
    n_reads: np.ndarray        # int32 per read id
    no_clusters: bool          # main.py:247-249 early return ("No clusters were found.")
    stats: dict
    edges: EdgeList = None     # the similarity graph, when the call asked for it (edges=True)


class DeviceTable:
    """The table's columns resident in HBM (torch tensors own the memory)."""

    def __init__(self, table: ColumnarTable, device, order=None):
        self.n_rows, self.n_reads = table.n_rows, table.n_reads
        self.cols = {k: torch.from_numpy(np.ascontiguousarray(getattr(table, k), dtype=np.int32)).to(device) for k in _COLS}
        self.order = None
        if order is not None:
            self.order = torch.from_numpy(np.ascontiguousarray(order, dtype=np.int32)).to(device)
        self.out_cluster = torch.empty(max(self.n_reads, 1), dtype=torch.int32, device=device)
        self.out_n_reads = torch.empty(max(self.n_reads, 1), dtype=torch.int32, device=device)


_TABLE_ORDER = object()          # run_resident / _table default: the `order` the table object carries


NARROW_OF = {"chrom": ("chrom_u8", np.uint8), "n_alignments": ("n_alignments_u16", np.uint16), "rend": ("rspan_i16", np.int16),
             "qstart": ("qstart_u16", np.uint16), "qend": ("qend_u16", np.uint16)}


class PinnedTable:
    """The table's columns in pinned host memory (the e2e path copies them in every call).  compact=True stores the table in
    its WIRE FORMAT, 13.25 instead of 32 bytes per row over PCIe / NVLink: `chrom` as uint8, `n_alignments`, `qstart`, `qend` as
    uint16 and `rend` as the int16 difference to `rstart` when the values fit, no `aln_size` when it equals qend - qstart on
    every row (what collect_mapping_info.py:88 writes), and run lengths instead of `read_id` when the rows of every read are
    contiguous and in id order.  Every identity is verified here before it is relied on; the library widens on the device."""

    def __init__(self, table: ColumnarTable, order=None, compact=False):
        self.n_rows, self.n_reads = table.n_rows, table.n_reads
        self.cols, self.narrow = {}, {}
        n = self.n_rows

        def pin(a):
            return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        if compact and n > 0:
            i64 = {k: np.asarray(getattr(table, k), dtype=np.int64) for k in ("chrom", "n_alignments", "rstart", "rend", "qstart", "qend")}
            if table.n_chrom <= 256 and i64["chrom"].min() >= 0:
                self.narrow["chrom_u8"] = pin(i64["chrom"].astype(np.uint8))
            if 0 <= i64["n_alignments"].min() and i64["n_alignments"].max() < 65536:
                self.narrow["n_alignments_u16"] = pin(i64["n_alignments"].astype(np.uint16).view(np.int16))
            span = i64["rend"] - i64["rstart"]
            if -32768 <= span.min() and span.max() < 32768:
                self.narrow["rspan_i16"] = pin(span.astype(np.int16))
            if 0 <= i64["qstart"].min() and i64["qstart"].max() < 65536 and 0 <= i64["qend"].min() and i64["qend"].max() < 65536:
                self.narrow["qstart_u16"] = pin(i64["qstart"].astype(np.uint16).view(np.int16))
                self.narrow["qend_u16"] = pin(i64["qend"].astype(np.uint16).view(np.int16))
        self.aln_is_qspan = bool(compact and n > 0 and np.array_equal(
            np.asarray(table.aln_size, dtype=np.int64), np.asarray(table.qend, dtype=np.int64) - np.asarray(table.qstart, dtype=np.int64)))
        self.rows_per_read = None
        if compact and n > 0:                                # rows of a read contiguous, reads in id order: send run lengths
            rid = np.asarray(table.read_id)
            cnt = np.bincount(rid, minlength=self.n_reads)
            if cnt.min(initial=1) >= 1 and cnt.max(initial=0) <= 255 and np.array_equal(rid, np.repeat(np.arange(self.n_reads, dtype=rid.dtype), cnt)):
                self.rows_per_read = pin(cnt.astype(np.uint8))
        for k in _COLS:
            if (k in NARROW_OF and NARROW_OF[k][0] in self.narrow) or (k == "aln_size" and self.aln_is_qspan) or \
                    (k == "read_id" and self.rows_per_read is not None):
                continue
            t = torch.empty(max(n, 1), dtype=torch.int32).pin_memory()
            t[:n] = torch.from_numpy(np.ascontiguousarray(getattr(table, k), dtype=np.int32))
            self.cols[k] = t
        self.order = None
        if order is not None:
            self.order = torch.from_numpy(np.ascontiguousarray(order, dtype=np.int32)).pin_memory()
        self.out_cluster = torch.empty(max(self.n_reads, 1), dtype=torch.int32).pin_memory()
        self.out_n_reads = torch.empty(max(self.n_reads, 1), dtype=torch.int32).pin_memory()

    def wire_columns(self):
        """name -> (host tensor, number of valid elements): everything that crosses PCIe for this table."""
        out = {k: (v, self.n_rows) for k, v in self.cols.items()}
        out.update({k: (v, self.n_rows) for k, v in self.narrow.items()})
        if self.rows_per_read is not None:
            out["rows_per_read_u8"] = (self.rows_per_read, self.n_reads)
        return out

    @property
    def h2d_bytes(self):
        return sum(n * t.element_size() for t, n in self.wire_columns().values()) + \
            (4 * int(self.order.numel()) if self.order is not None else 0)

    @property
    def d2h_bytes(self):
        return 8 * self.n_reads


class DeviceWireTable:
    """Multi-GPU ingest of HOST columns: the table's wire columns on this rank's device, filled by `upload`: every rank copies
    only its 1/world slice of every column over its own PCIe link straight into place and one in-place all-gather per column
    over NVLink completes it (no staging buffer, no extra pass).  The library widens the narrow columns on the device
    (fslrc_mg_prepare accepts them as they are)."""

    def __init__(self, ptab: PinnedTable, device, world):
        from .sharded import row_slice
        self.n_rows, self.n_reads = ptab.n_rows, ptab.n_reads
        self.aln_is_qspan, self.order = ptab.aln_is_qspan, None
        self.world, self.device = world, device
        self.wire = {}
        for k, (t, n) in ptab.wire_columns().items():
            chunk = row_slice(n, 0, world)[2]
            self.wire[k] = (torch.zeros(max(chunk * world, 1), dtype=t.dtype, device=device), n)
        self.cols = {k: v[0] for k, v in self.wire.items() if k in _COLS}
        self.narrow = {k: v[0] for k, v in self.wire.items() if k not in _COLS and k != "rows_per_read_u8"}
        self.rows_per_read = self.wire["rows_per_read_u8"][0] if "rows_per_read_u8" in self.wire else None
        self.out_cluster = torch.empty(max(self.n_reads, 1), dtype=torch.int32, device=device)
        self.out_n_reads = torch.empty(max(self.n_reads, 1), dtype=torch.int32, device=device)

    def upload(self, ptab: PinnedTable, rank, world, group=None):
        from .sharded import gather_column_inplace
        for k, (src, n) in ptab.wire_columns().items():
            gather_column_inplace(src, self.wire[k][0], n, rank, world, group)


class _DevView:
    """Device memory owned by the library, exposed to torch through __cuda_array_interface__ (int32)."""

    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<i4", "data": (int(ptr), False), "version": 2}


class ResidentTable:
    """A mappings table built on the device and kept there by the library context (tsv.ParsedBed, mapping_info.BamTable).
    Quacks like ColumnarTable where the engine needs it.  The context holds ONE table of each kind: the next open on the
    same engine frees this one's device columns, after which every method raises RuntimeError ("stale")."""

    _replaced = ""          # subclasses: what replaced a stale table, for the error message
    _names_fn = ""          # subclasses: the library's qname entry point, fn(ctx, offsets, lengths)
    _close_fn = ""          # subclasses: the library's close

    def __init__(self, engine, data, info):
        self.engine, self._data, self.info = engine, data, info
        self.n_rows, self.n_reads = int(info.n_rows), int(info.n_reads)
        self.order = None
        self.out_cluster = torch.empty(max(self.n_reads, 1), dtype=torch.int32, device=engine.device)
        self.out_n_reads = torch.empty(max(self.n_reads, 1), dtype=torch.int32, device=engine.device)
        self._names = None
        gen = engine._table_gen
        gen[type(self)] = self._gen = gen.get(type(self), 0) + 1

    def _live(self):
        if self.engine is None:
            raise RuntimeError("%s is closed" % type(self).__name__)
        if self._gen != self.engine._table_gen[type(self)]:
            raise RuntimeError("stale %s: %s (the library context holds one at a time)" % (type(self).__name__, self._replaced))

    @property
    def n_chrom(self):
        return len(self.chrom_names)

    def _name_bytes(self):
        """The bytes the offsets of the names entry point index."""
        raise NotImplementedError

    def qnames(self):
        """qname of every read id (ParsedBed: ids in order of first appearance; BamTable: in output order), sliced out of
        the input bytes on the host."""
        if self._names is None:
            self._live()
            off = np.zeros(max(self.n_reads, 1), dtype=np.int64)
            ln = np.zeros(max(self.n_reads, 1), dtype=np.int32)
            self.engine._check(getattr(self.engine.lib, self._names_fn)(self.engine.ctx, off.ctypes.data, ln.ctypes.data))
            buf = self._name_bytes()
            self._names = np.array([buf[o:o + l].decode() for o, l in zip(off[:self.n_reads], ln[:self.n_reads])], dtype=object)
        return self._names

    def cluster(self, cluster_mask="subtelomere", tie_order=None, edges=False, **options):
        """The clustering step (main.py:209-257,334-342) on the device-resident table.  Returns ClusterResult; the per-read
        result also stays on the device (out_cluster / out_n_reads) for the renderers.
        tie_order: how fillings with equal starts are ordered (cluster.py:114), which decides the cluster numbering.
        None: `self.order` when the caller set one, else the GPU's stable sort (ties keep bed order).  "stable": the GPU's
        stable sort.  "reference": the permutation fslr's own `sort_values('start')` gives on this host, so the ids equal
        fslr's: the start column is built on the device (fslrc_filling_starts), sorted on the host with the reference's
        pandas call and sent back, once per table (kept for later calls); it applies to that call only.
        edges=True: ClusterResult.edges holds the similarity graph (cluster.py:187-227's match_df rows, as read ids); for a
        ParsedBed, edges_bytes() / write_edges() can render it until the next clustering call on this engine."""
        self._live()
        params = ClusterParams.from_options(self, cluster_mask=cluster_mask, **options)
        out = self.engine.run_resident(self, self, params, order=self.engine.tie_order(self, tie_order), edges=edges)
        stats, el = out if edges else (out, None)
        n = self.n_reads
        return ClusterResult(self.out_cluster[:n].cpu().numpy(), self.out_n_reads[:n].cpu().numpy(), bool(stats["no_clusters"]), stats, el)

    def close(self):
        if self.engine is not None:
            if self._gen == self.engine._table_gen[type(self)]:    # (a stale object owns nothing any more)
                getattr(self.engine.lib, self._close_fn)(self.engine.ctx)
            self.engine = None


class Engine:
    def __init__(self, device=0):
        if not torch.cuda.is_available():
            raise RuntimeError("fslr_b200: no CUDA device — this package has no CPU fallback")
        self.lib = _native.load()
        self.device = torch.device("cuda", device)
        torch.cuda.set_device(self.device)
        torch.zeros(1, device=self.device)            # make sure the primary context exists
        self.ctx = C.c_void_p()
        rc = self.lib.fslrc_create(device, C.byref(self.ctx))
        if rc != 0:
            raise _native.FslrError(rc, "fslrc_create failed")
        self._capture = False
        self._table_gen = {}                          # ResidentTable subclass -> generation of the table the context holds

    def pinned_bytes(self, n):
        """A pinned uint8 staging buffer of at least n bytes, kept and reused (pinning hundreds of MB costs more than the
        copy it speeds up).  The returned view is valid until the next call."""
        buf = getattr(self, "_pinned", None)
        if buf is None or buf.numel() < n:
            self._pinned = buf = torch.empty(max(int(n * 1.25), 1 << 20), dtype=torch.uint8).pin_memory()
        return buf[:max(n, 1)]

    def _cuda_stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def open_table(self, fn, args, hash_seed, info):
        """fn(ctx, *args, seed, &info, stream): an open of a device-resident table, called again with the next seed (up to
        four seeds) when two names share a 64-bit hash."""
        for attempt in range(4):
            rc = fn(self.ctx, *args, hash_seed + attempt, C.byref(info), self._cuda_stream())
            if rc != _native.ERR_HASH_COLLISION:
                break
        self._check(rc)

    def render_bytes(self, fn, *args):
        """fn(ctx, *args, out, cap, &n_out, stream): a renderer of a device-resident table, called once for the size and once
        into the reused pinned staging buffer.  Returns a VIEW of that buffer: valid until the next rendering call."""
        n = C.c_int64()
        self._check(fn(self.ctx, *args, None, 0, C.byref(n), self._cuda_stream()))
        out = self.pinned_bytes(n.value)
        self._check(fn(self.ctx, *args, out.data_ptr(), n.value, C.byref(n), self._cuda_stream()))
        return out[:n.value].numpy()

    def close(self):
        if getattr(self, "ctx", None):
            self.lib.fslrc_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- argument marshalling
    def _params(self, table, params: ClusterParams):
        p = _native.Params()
        p.overlap = float(params.overlap)
        p.qlen_c = 1 - params.qlen_diff                 # cluster.py:179
        p.naln_c = 1 - params.n_alignment_diff          # cluster.py:181
        um = umax_table(list(params.jaccard_cutoffs))
        for i, v in enumerate(um):
            p.umax[i] = int(v)
        p.edge_threshold = int(max(min(params.edge_threshold, 2**62), -2**62))
        self._clen = np.ascontiguousarray(table_chrom_len(table), dtype=np.int64)
        m = params.chrom_masked if params.chrom_masked is not None else np.zeros(len(self._clen), np.uint8)
        self._cmask = np.ascontiguousarray(m, dtype=np.uint8)
        p.n_chrom = len(self._clen)
        p.chrom_len = self._clen.ctypes.data if len(self._clen) else None
        p.chrom_masked = self._cmask.ctypes.data if len(self._cmask) else None
        p.mask_subtelomere = int(bool(params.mask_subtelomere))
        p.subtel = int(params.subtel)
        return p

    @staticmethod
    def _table(buf, order=_TABLE_ORDER):
        t = _native.Table()
        t.n_rows, t.n_reads = buf.n_rows, buf.n_reads
        for k in _COLS:
            setattr(t, k, buf.cols[k].data_ptr() if k in buf.cols else None)
        narrow = getattr(buf, "narrow", None) or {}
        for k in ("chrom_u8", "n_alignments_u16", "rspan_i16", "qstart_u16", "qend_u16"):
            setattr(t, k, narrow[k].data_ptr() if k in narrow else None)
        t.aln_size_is_qspan = int(bool(getattr(buf, "aln_is_qspan", False)))
        rpr = getattr(buf, "rows_per_read", None)
        t.rows_per_read_u8 = rpr.data_ptr() if rpr is not None else None
        if order is _TABLE_ORDER:
            order = buf.order
        if order is not None:
            t.order, t.n_order = order.data_ptr(), int(order.numel())
        else:
            t.order, t.n_order = None, 0
        return t

    def _check(self, rc):
        if rc != 0:
            raise _native.FslrError(rc, self.lib.fslrc_last_error(self.ctx).decode())

    # ---- edge capture (fslrc_set_edge_capture)
    def _set_capture(self, on):
        """A call with edges=True switches capture on and leaves it on, so that the list stays in the context for the
        renderer (ParsedBed.edges_bytes); the next call without edges switches it off first (which frees the list)."""
        if bool(on) != self._capture:
            self._check(self.lib.fslrc_set_edge_capture(self.ctx, int(bool(on))))
            self._capture = bool(on)

    def edge_list(self):
        """The edge list the last clustering call captured (fslrc_edges), as host arrays."""
        n = C.c_int64()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        self._check(self.lib.fslrc_edges(self.ctx, None, None, None, 0, C.byref(n), C.c_void_p(stream)))
        m = max(n.value, 1)
        r1 = torch.empty(m, dtype=torch.int32, device=self.device)
        r2 = torch.empty(m, dtype=torch.int32, device=self.device)
        jac = torch.empty(m, dtype=torch.float64, device=self.device)
        self._check(self.lib.fslrc_edges(self.ctx, r1.data_ptr(), r2.data_ptr(), jac.data_ptr(), m, C.byref(n), C.c_void_p(stream)))
        k = n.value
        return EdgeList(r1[:k].cpu().numpy(), r2[:k].cpu().numpy(), jac[:k].cpu().numpy())

    # ---- compute entry points
    def run_resident(self, dtab: DeviceTable, chrom_table, params: ClusterParams, order=_TABLE_ORDER, edges=False):
        """Inputs already in HBM; outputs stay in HBM (dtab.out_cluster / out_n_reads).  Returns stats dict, or
        (stats, EdgeList) with edges=True (the similarity graph of this call, which also stays in the context until the
        next clustering call).
        order: the tie permutation of this call only (device int32 [n_fillings]; None = the GPU's stable sort); by default
        dtab.order."""
        p = self._params(chrom_table, params)
        t = self._table(dtab, order)
        st = _native.Stats()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        self._set_capture(edges)
        self._check(self.lib.fslrc_cluster_device(self.ctx, C.byref(t), C.byref(p), dtab.out_cluster.data_ptr(),
                                                  dtab.out_n_reads.data_ptr(), C.byref(st), C.c_void_p(stream)))
        if edges:
            return st.as_dict(self.lib), self.edge_list()
        return st.as_dict(self.lib)

    def filling_starts(self, dtab):
        """The `start` column cluster.py:114 sorts (fslrc_filling_starts), computed on the device from dtab's device
        columns: a device int32 tensor [n_fillings]."""
        out = torch.empty(max(dtab.n_rows, 1), dtype=torch.int32, device=self.device)
        n = C.c_int64()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        self._check(self.lib.fslrc_filling_starts(self.ctx, C.byref(self._table(dtab, None)), out.data_ptr(), out.numel(),
                                                  C.byref(n), C.c_void_p(stream)))
        return out[:n.value]

    def reference_order(self, dtab):
        """The reference's tie permutation (cluster.py:114) for a device-resident table (ParsedBed, BamTable): the start
        column from the device, sorted on the host by cluster.reference_order_of_starts (numpy's unstable sort, whose tie
        order is this host's), uploaded as the device int32 `order` fslrc_cluster_device takes."""
        from .cluster import reference_order_of_starts
        start = self.filling_starts(dtab).cpu().numpy()
        return torch.from_numpy(reference_order_of_starts(start)).to(self.device)

    def tie_order(self, dtab, tie_order):
        """The `order` run_resident gets for ParsedBed / BamTable.cluster(tie_order=...): None = dtab.order as set by the
        caller (else stable), "stable" = the GPU's stable sort, "reference" = reference_order(dtab), computed once and kept
        on the table (dtab._reference_order; the table does not change after it is built)."""
        if tie_order is None:
            return dtab.order
        if tie_order == "stable":
            return None
        if tie_order == "reference":
            if getattr(dtab, "_reference_order", None) is None:
                dtab._reference_order = self.reference_order(dtab)
            return dtab._reference_order
        raise ValueError("tie_order must be None, 'stable' or 'reference', not %r" % (tie_order,))

    def run_host(self, ptab: PinnedTable, chrom_table, params: ClusterParams, edges=False):
        """Host buffers in, host buffers out (H2D + D2H inside the call).  Returns stats dict.  edges: capture the
        similarity graph (read it with edge_list())."""
        p = self._params(chrom_table, params)
        t = self._table(ptab)
        st = _native.Stats()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        self._set_capture(edges)
        self._check(self.lib.fslrc_cluster_host(self.ctx, C.byref(t), C.byref(p), ptab.out_cluster.data_ptr(),
                                                ptab.out_n_reads.data_ptr(), C.byref(st), C.c_void_p(stream)))
        return st.as_dict(self.lib)

    def cluster(self, table: ColumnarTable, params: ClusterParams, order=None, edges=False) -> ClusterResult:
        """edges=True: ClusterResult.edges holds the similarity graph of this call."""
        ptab = PinnedTable(table, order)
        stats = self.run_host(ptab, table, params, edges=edges)
        n = table.n_reads
        return ClusterResult(ptab.out_cluster[:n].numpy().copy(), ptab.out_n_reads[:n].numpy().copy(),
                             bool(stats["no_clusters"]), stats, self.edge_list() if edges else None)

    # ---- multi-GPU: pair space sharded over ranks, three exchange steps (SURVEY §8e)
    def run_sharded(self, dtab: DeviceTable, chrom_table, params: ClusterParams, rank, world, group=None):
        """Every rank holds the whole table in HBM (dtab); candidate generation and the pair tests run on shard `rank` of `world`.
        Exchange steps (torch.distributed, NCCL on GPUs): sum-all-reduce of the per-read partner counters (4 bytes per query
        read), all-gather of the recorded pairs of saturating reads (8 bytes per pair: the replay needs them on every
        rank), all-gather of each rank's spanning forest.  Every rank ends with the full result in dtab.out_*."""
        import os
        import time
        from .sharded import exchange_counts, exchange_forests
        dbg = os.environ.get("FSLRC_DEBUG_MG") == "1"
        tl = []

        def lap(name):
            if dbg:
                torch.cuda.synchronize()
                tl.append((name, time.perf_counter()))
        p = self._params(chrom_table, params)
        t = self._table(dtab)
        st = _native.Stats()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        lap("start")
        self._check(self.lib.fslrc_mg_prepare(self.ctx, C.byref(t), C.byref(p), C.c_void_p(stream)))
        lap("prepare")
        ptr, n = C.c_void_p(), C.c_int64()
        self._check(self.lib.fslrc_mg_pair(self.ctx, rank, world, C.byref(ptr), C.byref(n)))
        lap("pair")
        if n.value > 0 and world > 1:
            exchange_counts(torch.as_tensor(_DevView(ptr.value, (n.value,)), device=self.device), group)
        lap("allreduce_counters")
        self._check(self.lib.fslrc_mg_partners(self.ctx, rank, world, C.byref(ptr), C.byref(n)))
        lap("partners")
        npairs = int(n.value)
        if world > 1:
            local = (torch.as_tensor(_DevView(ptr.value, (2 * npairs,)), device=self.device) if npairs > 0
                     else torch.zeros(0, dtype=torch.int32, device=self.device))
            pairs, per_rank = exchange_forests(local, group)                   # (same variable-length all-gather)
            npairs = int(sum(per_rank))
            pptr = pairs.data_ptr() if npairs > 0 else None
        else:
            pptr = ptr.value if npairs > 0 else None
        lap("allgather_pairs")
        self._check(self.lib.fslrc_mg_replay(self.ctx, rank, world, pptr, npairs, C.byref(ptr), C.byref(n)))
        lap("replay_union")
        ne = int(n.value)
        if world > 1:
            local = (torch.as_tensor(_DevView(ptr.value, (2 * ne,)), device=self.device) if ne > 0
                     else torch.zeros(0, dtype=torch.int32, device=self.device))
            forest, per_rank = exchange_forests(local, group)
            tot = int(sum(per_rank))
            fptr = forest.data_ptr() if tot > 0 else None
        else:
            tot, fptr = ne, ptr.value if ne > 0 else None
        lap("allgather_forests")
        self._check(self.lib.fslrc_mg_finish(self.ctx, fptr, tot, dtab.out_cluster.data_ptr(), dtab.out_n_reads.data_ptr(),
                                             C.byref(st)))
        lap("finish")
        if dbg and rank == 0:
            import sys
            print("[mg] " + "  ".join("%s %.2f" % (b[0], 1e3 * (b[1] - a[1])) for a, b in zip(tl, tl[1:])) + "  (ms; pairs %d, forest edges %d)" % (npairs, tot),
                  file=sys.stderr)
        return st.as_dict(self.lib)

    def choose_alignment(self, read_id, alignment_score, cluster, n_clusters):
        """cluster.py:237-254 on the GPU.  read_id/alignment_score: int32 per table row; cluster: int32 per read (dense ids).
        Returns (is_rep uint8 [n_reads], rep_read int32 [n_clusters])."""
        rid = np.ascontiguousarray(read_id, dtype=np.int32)
        sc = np.ascontiguousarray(alignment_score, dtype=np.int32)
        cl = np.ascontiguousarray(cluster, dtype=np.int32)
        is_rep = np.zeros(max(cl.shape[0], 1), dtype=np.uint8)
        rep = np.full(max(int(n_clusters), 1), -1, dtype=np.int32)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        self._check(self.lib.fslrc_choose_alignment_host(self.ctx, rid.shape[0], cl.shape[0], int(n_clusters), rid.ctypes.data,
                                                         sc.ctypes.data, cl.ctypes.data, is_rep.ctypes.data, rep.ctypes.data,
                                                         C.c_void_p(stream)))
        return is_rep[:cl.shape[0]], rep[:int(n_clusters)]

    def launch_count(self):
        return int(self.lib.fslrc_launch_count(self.ctx))

    def int_peak(self):
        v = C.c_double()
        self._check(self.lib.fslrc_int_peak(self.ctx, C.byref(v)))
        return v.value


class HostPipeline:
    """Host-buffer clustering of a stream of tables with the upload of one table overlapping the kernels of the previous
    one: `depth` library contexts, each with its own CUDA stream and worker thread (the C ABI call blocks its thread, not the
    interpreter).  This is how a service clusters sample after sample; `bench.py` uses it for the end-to-end number."""

    def __init__(self, device=0, depth=2, blocking_sync=None):
        import os
        from concurrent.futures import ThreadPoolExecutor
        self.engines = [Engine(device) for _ in range(depth)]
        if blocking_sync is None:                          # default: sleep in the waits — spinning worker threads starve each other
            blocking_sync = os.environ.get("FSLR_B200_BLOCKING_SYNC", "1") == "1"   # on hosts that give the process few cores
        for e in self.engines:                            # worker threads sleep in their waits instead of spinning
            e.lib.fslrc_set_blocking_sync(e.ctx, int(bool(blocking_sync)))
        self.streams = [torch.cuda.Stream(device=self.engines[0].device) for _ in range(depth)]
        self.pool = ThreadPoolExecutor(max_workers=depth)
        self.depth, self._next = depth, 0
        import threading
        self._locks = [threading.Lock() for _ in range(depth)]    # a library context is not re-entrant

    def _run(self, slot, ptab, chrom_table, params):
        eng, stream = self.engines[slot], self.streams[slot]
        torch.cuda.set_device(eng.device)
        with self._locks[slot]:
            p = eng._params(chrom_table, params)
            t = eng._table(ptab)
            st = _native.Stats()
            eng._check(eng.lib.fslrc_cluster_host(eng.ctx, C.byref(t), C.byref(p), ptab.out_cluster.data_ptr(),
                                                  ptab.out_n_reads.data_ptr(), C.byref(st), C.c_void_p(stream.cuda_stream)))
            return st.as_dict(eng.lib)

    def _run_resident(self, slot, dtab, chrom_table, params):
        eng, stream = self.engines[slot], self.streams[slot]
        torch.cuda.set_device(eng.device)
        with self._locks[slot]:
            p = eng._params(chrom_table, params)
            t = eng._table(dtab)
            st = _native.Stats()
            eng._check(eng.lib.fslrc_cluster_device(eng.ctx, C.byref(t), C.byref(p), dtab.out_cluster.data_ptr(),
                                                    dtab.out_n_reads.data_ptr(), C.byref(st), C.c_void_p(stream.cuda_stream)))
            return st.as_dict(eng.lib)

    def submit_resident(self, dtab: DeviceTable, chrom_table, params):
        """Same for a table that already lives in HBM (results stay in dtab.out_*): the latency-bound replay of one table
        runs beside the issue-bound kernels of the next."""
        slot = self._next
        self._next = (self._next + 1) % self.depth
        return self.pool.submit(self._run_resident, slot, dtab, chrom_table, params)

    def submit(self, ptab: PinnedTable, chrom_table, params):
        """ptab must not be reused by another submit before this one's future is done (its out_* buffers receive the result)."""
        slot = self._next
        self._next = (self._next + 1) % self.depth
        return self.pool.submit(self._run, slot, ptab, chrom_table, params)

    def launch_count(self):
        return sum(e.launch_count() for e in self.engines)

    def close(self):
        self.pool.shutdown(wait=True)
        for e in self.engines:
            e.close()


def table_chrom_len(table):
    return table.chrom_len


_engines = {}


def get_engine(device=0):
    if device not in _engines:
        _engines[device] = Engine(device)
    return _engines[device]
