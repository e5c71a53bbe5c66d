"""`<base>.mappings.bed` in and `<base>.mappings.cluster.bed` out on the GPU (SURVEY.md §8f row 1).

`read_mappings_bed(path)` replaces `pd.read_csv(path, sep='\\t')` + factorisation (/root/reference/fslr/main.py:209 and the
host side of fslr_b200.table.ColumnarTable.from_dataframe): the raw bytes go to the device once, the columnar table is
built there (fslrc_tsv_open) and stays there, so the clustering step runs on it without any further host<->device
traffic.  `ParsedBed.write_cluster_bed` renders the reference's output file (main.py:334-349): every input line plus the
float `cluster` / `n_reads` columns; `ParsedBed.write_representative_bed` the second one (main.py:351-352): the lines of
each cluster's representative read plus those columns and `avg_alignment_score`.  There is no CPU path: these functions raise without the CUDA library or a device.
"""
import ctypes as C

import numpy as np
import torch

from . import _native
from .engine import ClusterResult, DeviceTable, _DevView, get_engine
from .table import ClusterParams

_COLS = ("read_id", "chrom", "rstart", "rend", "aln_size", "qstart", "qend", "n_alignments")


class ParsedBed:
    """A mappings table parsed on the device.  Quacks like ColumnarTable where the engine needs it (chrom_names, chrom_len,
    n_chrom, n_rows, n_reads); the columns are device tensors that alias memory owned by the library context."""

    def __init__(self, engine, data, info, chrom_names, chr_lengths):
        self.engine, self._data, self.info = engine, data, info
        self.n_rows, self.n_reads = int(info.n_rows), int(info.n_reads)
        self.chrom_names = chrom_names
        self.chrom_len = np.array([int((chr_lengths or {}).get(c, 0) or 0) for c in chrom_names], dtype=np.int64)
        self.parse_ms = float(info.parse_ms)
        self.filter_ms = float(info.filter_ms)
        dev = engine.device
        view = lambda p: (torch.as_tensor(_DevView(p, (self.n_rows,)), device=dev) if self.n_rows > 0 and p
                          else torch.zeros(0, dtype=torch.int32, device=dev))
        self.cols = {k: view(getattr(info, k)) for k in _COLS}
        self.alignment_score = view(info.alignment_score) if info.has_score else None
        self.order = None
        self.out_cluster = torch.empty(max(self.n_reads, 1), dtype=torch.int32, device=dev)
        self.out_n_reads = torch.empty(max(self.n_reads, 1), dtype=torch.int32, device=dev)
        self._names = None
        # the library context keeps ONE parsed table (fslrc_tsv_open frees the previous one): a later read_mappings_bed on the
        # same engine invalidates this object, whose device columns would then point at freed memory
        engine._tsv_gen = getattr(engine, "_tsv_gen", 0) + 1
        self._gen = engine._tsv_gen

    def _live(self):
        if self.engine is None:
            raise RuntimeError("ParsedBed is closed")
        if self._gen != self.engine._tsv_gen:
            raise RuntimeError("stale ParsedBed: a later read_mappings_bed() on this device replaced the parsed table "
                               "(the library context holds one at a time)")

    @property
    def n_chrom(self):
        return len(self.chrom_names)

    def column(self, name):
        """Host copy of one parsed column (int32)."""
        self._live()
        t = self.alignment_score if name == "alignment_score" else self.cols[name]
        return t.cpu().numpy()

    def qnames(self):
        """qname of every read id (order of first appearance), sliced out of the file bytes on the host."""
        if self._names is None:
            self._live()
            off = np.zeros(max(self.n_reads, 1), dtype=np.int64)
            ln = np.zeros(max(self.n_reads, 1), dtype=np.int32)
            self.engine._check(self.engine.lib.fslrc_tsv_read_names(self.engine.ctx, off.ctypes.data, ln.ctypes.data))
            buf = self._data.tobytes() if not isinstance(self._data, (bytes, bytearray)) else self._data
            self._names = np.array([buf[o:o + l].decode() for o, l in zip(off[:self.n_reads], ln[:self.n_reads])], dtype=object)
        return self._names

    def cluster(self, cluster_mask="subtelomere", tie_order=None, edges=False, **options):
        """The clustering step on the device-resident table.  Returns ClusterResult; the per-read result also stays on the
        device (out_cluster / out_n_reads) for write_cluster_bed.
        tie_order: how fillings with equal starts are ordered (cluster.py:114), which decides the cluster numbering.
        None: `self.order` when the caller set one, else the GPU's stable sort (ties keep bed order).  "stable": the GPU's
        stable sort.  "reference": the permutation fslr's own `sort_values('start')` gives on this host, so the ids equal
        fslr's: the start column is built on the device (fslrc_filling_starts), sorted on the host with the reference's
        pandas call and sent back, once per table (kept for later calls); it applies to that call only.
        edges=True: ClusterResult.edges holds the similarity graph (cluster.py:187-227's match_df rows, as read ids), and
        edges_bytes() / write_edges() can render it until the next clustering call on this engine."""
        self._live()
        params = ClusterParams.from_options(self, cluster_mask=cluster_mask, **options)
        out = self.engine.run_resident(self, self, params, order=self.engine.tie_order(self, tie_order), edges=edges)
        stats, el = out if edges else (out, None)
        n = self.n_reads
        return ClusterResult(self.out_cluster[:n].cpu().numpy(), self.out_n_reads[:n].cpu().numpy(), bool(stats["no_clusters"]), stats, el)

    def _render(self, entry):
        self._live()
        fn, ctx = getattr(self.engine.lib, entry), self.engine.ctx
        stream = C.c_void_p(torch.cuda.current_stream(self.engine.device).cuda_stream)
        n = C.c_int64()
        self.engine._check(fn(ctx, self.out_cluster.data_ptr(), self.out_n_reads.data_ptr(), None, 0, C.byref(n), stream))
        out = self.engine.pinned_bytes(n.value)       # reused staging buffer: the result is valid until the next rendering call
        self.engine._check(fn(ctx, self.out_cluster.data_ptr(), self.out_n_reads.data_ptr(), out.data_ptr(), n.value, C.byref(n), stream))
        return out[:n.value].numpy()

    def cluster_bed_bytes(self):
        """`<base>.mappings.cluster.bed` (main.py:349) as bytes, rendered on the device from out_cluster / out_n_reads.  The
        returned array is a VIEW of the engine's reused pinned staging buffer: valid until the next rendering call of any
        table on this engine (copy it, or write it out, before that)."""
        return self._render("fslrc_tsv_write_cluster_bed")

    def write_cluster_bed(self, path):
        self.cluster_bed_bytes().tofile(path)

    def representative_bed_bytes(self):
        """`<base>.mappings.representative.bed` (main.py:351-352, cluster.py:237-254) as bytes, rendered on the device from
        the parsed alignment_score column and out_cluster / out_n_reads: the lines of each cluster's representative read
        (highest mean alignment_score, first in the table on ties) plus `cluster`, `n_reads` and `avg_alignment_score`
        (repr of the mean, as pandas writes a float64).  Raises FslrError without an alignment_score column or for a
        cluster id outside [0, n_reads).  Like cluster_bed_bytes, a VIEW of the engine's reused pinned staging buffer."""
        return self._render("fslrc_tsv_write_representative_bed")

    def write_representative_bed(self, path):
        self.representative_bed_bytes().tofile(path)

    def edges_bytes(self):
        """The edge list of the last cluster(edges=True) call as match_df.to_csv(sep="\\t", index=False) writes it (header
        `query1\\tquery2\\tjaccard_similarity`, one line per edge: both qnames and repr of the Jaccard similarity), rendered on
        the device (fslrc_tsv_write_edges).  Raises FslrError when the last clustering call on this engine was not a
        cluster(edges=True) of this table.  Like cluster_bed_bytes, a VIEW of the engine's reused pinned staging buffer."""
        self._live()
        fn, ctx = self.engine.lib.fslrc_tsv_write_edges, self.engine.ctx
        stream = C.c_void_p(torch.cuda.current_stream(self.engine.device).cuda_stream)
        n = C.c_int64()
        self.engine._check(fn(ctx, None, 0, C.byref(n), stream))
        out = self.engine.pinned_bytes(n.value)
        self.engine._check(fn(ctx, out.data_ptr(), n.value, C.byref(n), stream))
        return out[:n.value].numpy()

    def write_edges(self, path):
        self.edges_bytes().tofile(path)

    def close(self):
        if self.engine is not None:
            if self._gen == self.engine._tsv_gen:             # (a stale object owns nothing any more)
                self.engine.lib.fslrc_tsv_close(self.engine.ctx)
            self.engine = None


def read_mappings_bed(path_or_bytes, chr_lengths=None, device=0, hash_seed=0, filter_false=False):
    """Parse `<base>.mappings.bed` on the GPU.  chr_lengths: {chrom name: length} (the BAM-header lookup of main.py:225).
    filter_false: --filter-false (main.py:229-230), on the device: the reads whose qname contains "False" leave the table
    (fslrc_tsv_delete_false), so n_rows, n_reads, the columns, qnames() and both rendered files describe the kept rows.
    Chromosome ids and names stay those of the whole file, as main.py numbers them before it filters; malformed rows of
    dropped reads still raise, as pandas reads every row before delete_false runs."""
    eng = get_engine(device)
    if isinstance(path_or_bytes, (bytes, bytearray)):
        data = np.frombuffer(path_or_bytes, dtype=np.uint8)
    else:
        data = np.fromfile(path_or_bytes, dtype=np.uint8)
    info = _native.TsvInfo()
    stream = C.c_void_p(torch.cuda.current_stream(eng.device).cuda_stream)
    for attempt in range(4):                                            # a 64-bit hash collision between two names: reseed
        rc = eng.lib.fslrc_tsv_open(eng.ctx, data.ctypes.data, data.shape[0], hash_seed + attempt, C.byref(info), stream)
        if rc != _native.ERR_HASH_COLLISION:
            break
    eng._check(rc)
    if filter_false:
        eng._check(eng.lib.fslrc_tsv_delete_false(eng.ctx, C.byref(info), stream))
    names = []
    buf = C.create_string_buffer(4096)
    for c in range(info.n_chrom):
        n = eng.lib.fslrc_tsv_chrom_name(eng.ctx, c, buf, 4096)
        if n < 0:
            raise _native.FslrError(n, "fslrc_tsv_chrom_name")
        names.append(buf.value.decode())
    return ParsedBed(eng, data, info, names, chr_lengths)
