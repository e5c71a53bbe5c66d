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
from .engine import _COLS, ResidentTable, _DevView, get_engine


class ParsedBed(ResidentTable):
    """A mappings table parsed on the device.  Quacks like ColumnarTable where the engine needs it (chrom_names, chrom_len,
    n_chrom, n_rows, n_reads); the columns are device tensors that alias memory owned by the library context."""

    _replaced = "a later read_mappings_bed() on this device replaced the parsed table"
    _names_fn = "fslrc_tsv_read_names"
    _close_fn = "fslrc_tsv_close"

    def __init__(self, engine, data, info, chrom_names, chr_lengths):
        super().__init__(engine, data, info)
        self.chrom_names = chrom_names
        self.chrom_len = np.array([int((chr_lengths or {}).get(c, 0) or 0) for c in chrom_names], dtype=np.int64)
        self.parse_ms = float(info.parse_ms)
        self.filter_ms = float(info.filter_ms)
        dev = engine.device
        view = lambda p: (torch.as_tensor(_DevView(p, (self.n_rows,)), device=dev) if self.n_rows > 0 and p
                          else torch.zeros(0, dtype=torch.int32, device=dev))
        self.cols = {k: view(getattr(info, k)) for k in _COLS}
        self.alignment_score = view(info.alignment_score) if info.has_score else None

    def column(self, name):
        """Host copy of one parsed column (int32)."""
        self._live()
        t = self.alignment_score if name == "alignment_score" else self.cols[name]
        return t.cpu().numpy()

    def _name_bytes(self):
        return bytes(self._data)

    def _render(self, entry):
        self._live()
        return self.engine.render_bytes(getattr(self.engine.lib, entry), self.out_cluster.data_ptr(), self.out_n_reads.data_ptr())

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
        return self.engine.render_bytes(self.engine.lib.fslrc_tsv_write_edges)

    def write_edges(self, path):
        self.edges_bytes().tofile(path)


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
    eng.open_table(eng.lib.fslrc_tsv_open, (data.ctypes.data, data.shape[0]), hash_seed, info)
    if filter_false:
        eng._check(eng.lib.fslrc_tsv_delete_false(eng.ctx, C.byref(info), eng._cuda_stream()))
    names = []
    buf = C.create_string_buffer(4096)
    for c in range(info.n_chrom):
        n = eng.lib.fslrc_tsv_chrom_name(eng.ctx, c, buf, 4096)
        if n < 0:
            raise _native.FslrError(n, "fslrc_tsv_chrom_name")
        names.append(buf.value.decode())
    return ParsedBed(eng, data, info, names, chr_lengths)
