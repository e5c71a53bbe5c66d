"""`<base>.bwa_dodi.bam` -> `<base>.mappings.bed` on the GPU (SURVEY.md §8f row 4).

`mapping_info(f, outf, regions_path, primers)` has the signature and the output file of
/root/reference/fslr/collect_mapping_info.py:19-181 (called from main.py:181-183) without pysam: the BGZF blocks are
inflated on the DEVICE (fslr_b200/csrc/inflate.cuh: one warp per block, so only the compressed bytes cross PCIe; a host
zlib thread pool is the `device_inflate=False` alternative), the record boundaries are found there too, and everything else — CIGAR and aux parsing, grouping by read name, the primary record, the
strand flip of the query interval, the inferred primer rows of single-alignment reads, both sorts, short_anchor<50bp,
region overlaps, the TSV text with the decoded sequence — runs there (fslr_b200/csrc/bam.cuh).  The table stays on the
device, so `BamTable.cluster()` runs the clustering step on it without going through the file at all.
There is no CPU path: these functions raise without the CUDA library or a device.
"""
import ctypes as C
import struct
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch

from . import _native
from .engine import _COLS, ResidentTable, _DevView, get_engine

OUT_COLUMNS = ["chrom", "rstart", "rend", "qname", "n_alignments", "aln_size", "qstart", "qend", "strand", "mapq", "qlen",
               "alignment_score", "short_anchor<50bp", "fslr_version", "inferred_by_primer", "seq"]   # collect_mapping_info.py:176-177


def _bgzf_blocks(mv):
    """The blocks of the BGZF bytes `mv`, in file order, as (index, file offset, payload start, payload end, CRC32, ISIZE).
    A block is a gzip member whose `BC` extra subfield gives its size; the trailer holds CRC32 and ISIZE."""
    p, k = 0, 0
    while p < len(mv):
        if len(mv) - p < 18 or bytes(mv[p:p + 4]) != b"\x1f\x8b\x08\x04":
            raise ValueError("not a BGZF/BAM file (block header at byte %d)" % p)
        xlen = struct.unpack_from("<H", mv, p + 10)[0]
        q, bsize = p + 12, None
        while q < p + 12 + xlen:                                          # extra subfields: SI1 SI2 SLEN data
            si1, si2, slen = mv[q], mv[q + 1], struct.unpack_from("<H", mv, q + 2)[0]
            if si1 == 66 and si2 == 67 and slen == 2:
                bsize = struct.unpack_from("<H", mv, q + 4)[0] + 1
            q += 4 + slen
        if bsize is None or bsize < 12 + xlen + 8 or p + bsize > len(mv):
            raise ValueError("truncated BGZF block at byte %d" % p)
        crc, isize = struct.unpack_from("<II", mv, p + bsize - 8)
        yield k, p, p + 12 + xlen, p + bsize - 8, crc, isize
        p += bsize
        k += 1


def _inflate_block(mv, block):
    """One block of _bgzf_blocks inflated and checked against its trailer, as htslib checks it: the length against ISIZE,
    then the CRC-32 against CRC32.  A mismatch raises ValueError naming the block and its offset in the file."""
    k, p, s, e, crc, isize = block
    data = zlib.decompress(mv[s:e], -15)
    if len(data) != isize:
        raise ValueError("ISIZE mismatch in BGZF block %d (file offset %d): %d bytes inflated, ISIZE %d" % (k, p, len(data), isize))
    if zlib.crc32(data) != crc:
        raise ValueError("CRC32 mismatch in BGZF block %d (file offset %d)" % (k, p))
    return data


def inflate_bgzf(path_or_bytes, threads=8):
    """The uncompressed stream of a BGZF file as a uint8 array.  Block sizes come from the `BC` extra field and the ISIZE
    trailer, so every block inflates independently into its final place.  Every block is checked against its CRC32 and
    ISIZE; a mismatch raises ValueError naming the first bad block."""
    raw = path_or_bytes if isinstance(path_or_bytes, (bytes, bytearray, memoryview, np.ndarray)) else open(path_or_bytes, "rb").read()
    mv = memoryview(raw)
    blocks = list(_bgzf_blocks(mv))
    start = np.cumsum([0] + [b[5] for b in blocks])
    out = np.empty(int(start[-1]), dtype=np.uint8)

    def work(b):
        o = int(start[b[0]])
        out[o:o + b[5]] = np.frombuffer(_inflate_block(mv, b), dtype=np.uint8)

    if threads > 1 and len(blocks) > 4:
        with ThreadPoolExecutor(threads) as ex:
            list(ex.map(work, blocks, chunksize=64))                      # (results in block order: the first bad block raises)
    else:
        for b in blocks:
            work(b)
    return out


def bgzf_header_prefix(raw, want=None):
    """Inflate BGZF blocks from the start of `raw` (file bytes) until the BAM header — magic, text, reference list — is
    complete.  Returns (references, offset of the first alignment record in the inflated stream).  The blocks read are
    checked against their CRC32 and ISIZE (ValueError on a mismatch)."""
    mv = memoryview(raw)
    buf = bytearray()
    blocks = _bgzf_blocks(mv)

    def need(n):
        while len(buf) < n:
            b = next(blocks, None)
            if b is None:
                raise ValueError("truncated BAM header")
            buf.extend(_inflate_block(mv, b))

    need(12)
    if bytes(buf[:4]) != b"BAM\x01":
        raise ValueError("bad BAM magic")
    l_text = struct.unpack_from("<i", buf, 4)[0]
    need(12 + l_text)
    n_ref = struct.unpack_from("<i", buf, 8 + l_text)[0]
    q, refs = 12 + l_text, []
    for _ in range(n_ref):
        need(q + 4)
        l = struct.unpack_from("<i", buf, q)[0]
        need(q + 8 + l)
        refs.append((bytes(buf[q + 4:q + 4 + l - 1]).decode(), struct.unpack_from("<i", buf, q + 4 + l)[0]))
        q += 8 + l
    return refs, q


def parse_bam_header(buf):
    """(references [(name, length)], offset of the first alignment record) of an uncompressed BAM stream."""
    if buf.shape[0] < 12 or bytes(buf[:4]) != b"BAM\x01":
        raise ValueError("bad BAM magic")
    b = memoryview(buf)
    l_text = struct.unpack_from("<i", b, 4)[0]
    p = 8 + l_text
    n_ref = struct.unpack_from("<i", b, p)[0]
    p += 4
    refs = []
    for _ in range(n_ref):
        l = struct.unpack_from("<i", b, p)[0]
        refs.append((bytes(b[p + 4:p + 4 + l - 1]).decode(), struct.unpack_from("<i", b, p + 4 + l)[0]))
        p += 8 + l
    return refs, p


def read_regions(regions_path):
    """collect_mapping_info.py:28-36: {chrom: [(start, end)]}"""
    regions = {}
    if regions_path:
        with open(regions_path) as f:
            for line in f:
                l = line.strip().split("\t")
                regions.setdefault(l[0], []).append((int(l[1]), int(l[2])))
    return regions


def _default_version():
    try:
        from importlib.metadata import version
        return version("fslr")                                            # collect_mapping_info.py:20
    except Exception:                                                     # noqa: BLE001 - no installed fslr distribution
        from . import __version__
        return __version__


class BamTable(ResidentTable):
    """The mappings table built on the device from a BAM file, rows in the order of collect_mapping_info.py:174.  Quacks
    like ColumnarTable where the clustering engine needs it (chrom_names, chrom_len, n_chrom, n_rows, n_reads, cols)."""

    _replaced = "a later read_bam_table() on this device replaced the table"
    _names_fn = "fslrc_bam_read_names"
    _close_fn = "fslrc_bam_close"

    def __init__(self, engine, data, info, refs, primers, with_regions):
        super().__init__(engine, data, info)
        self.n_records, self.n_mapped = int(info.n_records), int(info.n_mapped)
        self.primer_names = list(primers)
        self.chrom_names = [n for n, _ in refs] + self.primer_names       # inferred rows carry the primer name as chrom (:124,143)
        self.chrom_len = np.array([l for _, l in refs] + [0] * len(self.primer_names), dtype=np.int64)
        self.with_regions = bool(with_regions)
        self.parse_ms = float(info.parse_ms)
        dev = engine.device
        view = lambda p: torch.as_tensor(_DevView(p, (self.n_rows,)), device=dev)
        self.columns = {k: view(getattr(info, k)) for k in _native.BAM_COLUMNS}
        self.cols = {k: self.columns[k] for k in _COLS}

    def column(self, name):
        """Host copy of one column (int32)."""
        self._live()
        return self.columns[name].cpu().numpy()

    def _stream(self):
        """The inflated BAM stream on the host (fetched from the device when the file was inflated there)."""
        if self._data is None:
            self._live()
            n = C.c_int64()
            self.engine._check(self.engine.lib.fslrc_bam_read_stream(self.engine.ctx, None, 0, C.byref(n)))
            self._data = np.empty(n.value, dtype=np.uint8)
            self.engine._check(self.engine.lib.fslrc_bam_read_stream(self.engine.ctx, self._data.ctypes.data, n.value, C.byref(n)))
        return self._data

    def _name_bytes(self):
        return self._stream().tobytes()

    def to_dataframe(self):
        """The table as pandas would read the written file back (without `seq` and `fslr_version`)."""
        import pandas as pd
        c = {k: self.column(k) for k in _native.BAM_COLUMNS}
        names = np.array(self.chrom_names, dtype=object)
        df = pd.DataFrame({"chrom": names[c["chrom"]], "rstart": c["rstart"], "rend": c["rend"], "qname": self.qnames()[c["read_id"]],
                           "n_alignments": c["n_alignments"], "aln_size": c["aln_size"], "qstart": c["qstart"], "qend": c["qend"],
                           "strand": np.where(c["strand"] != 0, "-", "+"), "mapq": c["mapq"], "qlen": c["qlen"],
                           "alignment_score": c["alignment_score"], "short_anchor<50bp": c["short_anchor"],
                           "inferred_by_primer": c["inferred_by_primer"]})
        if self.with_regions:
            ov = c["overlaps_region"].astype(np.float64)
            ov[ov < 0] = np.nan
            df["overlaps_region"] = ov if self.info.overlaps_as_float else ov.astype(np.int64)
        return df

    def mappings_bed_bytes(self, fslr_version=None):
        """`<base>.mappings.bed` (collect_mapping_info.py:176-181) as bytes, rendered on the device."""
        self._live()
        ver = (fslr_version if fslr_version is not None else _default_version()).encode()
        names = b"".join(n.encode() + b"\x00" for n in self.chrom_names)
        return self.engine.render_bytes(self.engine.lib.fslrc_bam_write_mappings_bed, names, ver)

    def write_mappings_bed(self, path, fslr_version=None):
        self.mappings_bed_bytes(fslr_version).tofile(path)


def read_bam_table(bam, regions_path=None, primers=None, device=0, hash_seed=0, threads=8, device_inflate=True):
    """Build the mappings table on the GPU.  bam: path or BGZF bytes (inflated on the device when device_inflate, else with
    zlib on `threads` host threads), or an already inflated uint8 array.
    primers: {name: sequence} (main.py hands the parsed primer file); only the sequence lengths are used (:133,151)."""
    eng = get_engine(device)
    inflated = isinstance(bam, np.ndarray)
    if inflated:
        data = np.ascontiguousarray(bam, dtype=np.uint8)
        refs, first = parse_bam_header(data)
    else:
        if isinstance(bam, (bytes, bytearray, memoryview)):
            raw = bam
        elif device_inflate:                                              # straight into the reused pinned staging buffer
            import os
            if os.path.getsize(bam) == 0:
                raise ValueError("%s: empty file" % bam)
            raw = eng.pinned_bytes(os.path.getsize(bam)).numpy()
            with open(bam, "rb") as f:
                if f.readinto(memoryview(raw)) != raw.shape[0]:
                    raise IOError("short read of %s" % bam)
        else:
            raw = np.fromfile(bam, dtype=np.uint8)
        if device_inflate:
            data = raw if isinstance(raw, np.ndarray) else np.frombuffer(raw, dtype=np.uint8)
            refs, first = bgzf_header_prefix(data)
        else:
            data = inflate_bgzf(raw, threads)
            refs, first = parse_bam_header(data)
            inflated = True
    primers = dict(primers or {})
    pnames = list(primers)
    if any(not n or "\x00" in n for n in pnames):
        raise ValueError("empty primer name")
    plen = np.array([len(primers[n]) for n in pnames], dtype=np.int32)
    regions = read_regions(regions_path)
    ref_id = {n: i for i, (n, _) in enumerate(refs)}
    rc, rs, re_ = [], [], []
    for chrom, iv in regions.items():
        if chrom in ref_id:
            for s, e in iv:
                rc.append(ref_id[chrom]); rs.append(s); re_.append(e)
    n_regions = len(rc) if regions else -1                               # `if regions:` (:72,96): an empty file means no column
    rc, rs, re_ = (np.asarray(a, dtype=np.int32) for a in (rc, rs, re_))
    info = _native.BamInfo()
    names = b"".join(n.encode() + b"\x00" for n in pnames)
    fn = eng.lib.fslrc_bam_open if inflated else eng.lib.fslrc_bam_open_bgzf
    eng.open_table(fn, (data.ctypes.data, data.shape[0], first, len(refs), names, plen.ctypes.data, len(pnames),
                        rc.ctypes.data, rs.ctypes.data, re_.ctypes.data, n_regions), hash_seed, info)
    return BamTable(eng, data if inflated else None, info, refs, pnames, n_regions >= 0)


def mapping_info(f, outf, regions_path, primers, fslr_version=None, device=0):
    """collect_mapping_info.mapping_info (collect_mapping_info.py:19): BAM `f` in, TSV `outf` out.  Returns the BamTable
    (still on the device) so that a caller can go on to `.cluster()` without re-reading `outf`."""
    t = read_bam_table(f, regions_path, primers, device=device)
    t.write_mappings_bed(outf, fslr_version)
    return t
