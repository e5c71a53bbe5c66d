"""The fast ingest (contiguous reads, no caller `order`) against the general ingest (FSLRC_GENERAL_INGEST=1) and the CPU
oracle, on the benchmark configurations at small scale and on tables built to hit the edges of the partition by chromosome
that carries the records: runs of equal (chrom, start) that straddle its tiles, runs too long for the tie window, one
chromosome and more chromosomes than one 8-bit digit, no intervals, 64 fillings in a read, a start beyond its chromosome's
length, and rows that violate the precondition."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _run(t, p, general):
    from fslr_b200.engine import get_engine
    old = os.environ.pop("FSLRC_GENERAL_INGEST", None)
    if general:
        os.environ["FSLRC_GENERAL_INGEST"] = "1"
    try:
        return get_engine(0).cluster(t, p)
    finally:
        os.environ.pop("FSLRC_GENERAL_INGEST", None)
        if old is not None:
            os.environ["FSLRC_GENERAL_INGEST"] = old


def _check(t, p):
    from oracle import oracle as orc
    fast, gen = _run(t, p, False), _run(t, p, True)
    ocl, onr, ost = orc.oracle_cluster(t, p)
    for res in (fast, gen):
        assert bool(ost["no_clusters"]) == res.no_clusters
        assert res.stats["n_intervals"] == ost["n_data"]
        if not res.no_clusters:
            assert np.array_equal(res.cluster, ocl)
            assert np.array_equal(res.n_reads, onr)
    return fast


def _table(reads, n_chrom, chrom_len):
    """reads: per read, a list of (chrom, start, end) fillings; every read gets a first and a last row around them."""
    from fslr_b200.table import ColumnarTable
    cols = {k: [] for k in ("read_id", "chrom", "rstart", "rend", "aln_size", "qstart", "qend", "n_alignments")}
    for r, fills in enumerate(reads):
        rows = [(0, 100, 600)] + list(fills) + [(0, 100, 600)]
        for j, (c, s, e) in enumerate(rows):
            cols["read_id"].append(r); cols["chrom"].append(c); cols["rstart"].append(s); cols["rend"].append(e)
            cols["aln_size"].append(500); cols["qstart"].append(500 * j); cols["qend"].append(500 * j + 500)
            cols["n_alignments"].append(len(rows))
    return ColumnarTable(**{k: np.asarray(v, np.int32) for k, v in cols.items()}, n_reads=len(reads),
                         chrom_names=["chr%d" % (c + 1) for c in range(n_chrom)],
                         chrom_len=np.full(n_chrom, chrom_len, np.int64))


def _paired_reads(n_pairs, n_chrom, n_starts, seed, fills=2):
    """Reads in pairs with the same starts and different ends: runs of equal (chrom, start) all over data order."""
    rng = np.random.default_rng(seed)
    reads = []
    for _ in range(n_pairs):
        f = [(int(rng.integers(n_chrom)), 2_000_000 + 1000 * int(rng.integers(n_starts)), 0) for _ in range(fills)]
        for _ in range(2):
            reads.append([(c, s, s + 400 + int(rng.integers(600))) for c, s, _ in f])
    return reads


@pytest.mark.parametrize("name,scale", [("C2", 1.0), ("C3", 0.05), ("C5", 0.02), ("C4", 0.02)])
def test_configs(name, scale):
    from fslr_b200 import synth
    from fslr_b200.table import ClusterParams, ColumnarTable
    t = ColumnarTable.from_synth(synth.make_config(name, scale))
    _check(t, ClusterParams.from_options(t, cluster_mask=synth.CONFIG_MASK[name]))


def test_tie_runs_straddle_partition_tiles():
    """~60k intervals on 3 chromosomes and 3000 starts: runs of up to ~25 equal (chrom, start), many cut by the 8192-item tiles."""
    from fslr_b200.table import ClusterParams
    t = _table(_paired_reads(15_000, 3, 3000, 1), 3, 10**8)
    res = _check(t, ClusterParams.from_options(t, edge_threshold=1))
    assert res.stats["n_intervals"] > 4 * 8192 and not res.no_clusters


def test_tie_run_longer_than_window():
    """60 reads on the same two intervals: a run of 60 equal (chrom, start) > TIE_WIN takes the three-sort order."""
    from fslr_b200.table import ClusterParams
    reads = _paired_reads(2000, 2, 500, 2) + [[(0, 5_000_000, 5_000_500 + k), (1, 6_000_000, 6_000_700 - k)] for k in range(60)]
    t = _table(reads, 2, 10**8)
    _check(t, ClusterParams.from_options(t, edge_threshold=2))


@pytest.mark.parametrize("n_chrom", [1, 256, 300])
def test_chromosome_counts(n_chrom):
    """One chromosome; 256 (one digit); 300 (two partition passes by chromosome)."""
    from fslr_b200.table import ClusterParams
    t = _table(_paired_reads(6000, n_chrom, 400, n_chrom, fills=3), n_chrom, 10**8)
    _check(t, ClusterParams.from_options(t, edge_threshold=1))


def test_no_intervals():
    from fslr_b200.table import ClusterParams
    t = _table([[] for _ in range(50)] + [[(0, 20_000, 20_500)]], 1, 10**8)
    p = ClusterParams.from_options(t, cluster_mask="chr1")
    res = _check(t, p)
    assert res.stats["n_intervals"] == 0


def test_read_with_64_fillings():
    from fslr_b200.table import ClusterParams
    big = [(0, 1_000_000 + 3000 * k, 1_000_800 + 3000 * k) for k in range(64)]
    reads = _paired_reads(500, 1, 300, 4) + [big, [(c, s, e + 7) for c, s, e in big]]
    t = _table(reads, 1, 10**8)
    res = _check(t, ClusterParams.from_options(t, edge_threshold=1))
    assert not res.no_clusters


def test_start_beyond_chromosome_length():
    """The fast ingest sorts on as many key bits as the chromosome lengths need; a start past them takes the general path."""
    from fslr_b200.table import ClusterParams
    reads = _paired_reads(500, 2, 9, 5)
    reads += [[(1, 5_000_000, 5_000_500)], [(1, 5_000_000, 5_000_450)]]                 # 22 key bits cover 4e6, not 5e6
    t = _table(reads, 2, 4_000_000)
    _check(t, ClusterParams.from_options(t, cluster_mask="", edge_threshold=1))


def test_rows_not_contiguous():
    """Rows of a read apart (EF_NONMONO): the fast ingest hands the table to the general path."""
    from fslr_b200.table import ClusterParams
    t = _table(_paired_reads(800, 2, 100, 6), 2, 10**8)
    perm = np.random.default_rng(6).permutation(t.n_rows)
    for k in ("read_id", "chrom", "rstart", "rend", "aln_size", "qstart", "qend", "n_alignments"):
        setattr(t, k, np.ascontiguousarray(getattr(t, k)[perm]))
    _, first = np.unique(t.read_id, return_index=True)
    order = np.argsort(first)
    remap = np.empty_like(order); remap[order] = np.arange(order.size)
    t.read_id = remap[t.read_id].astype(np.int32)
    _check(t, ClusterParams.from_options(t, edge_threshold=1))


def test_wire_format_host_call_c4():
    """The host call with the wire format uploads n_alignments last, on a second stream (tables of >= 2^20 rows, hence C4 at
    3 %), and the ingest waits for it before its first reader."""
    from fslr_b200 import synth
    from fslr_b200.engine import PinnedTable, get_engine
    from fslr_b200.table import ClusterParams, ColumnarTable
    from oracle import oracle as orc
    t = ColumnarTable.from_synth(synth.make_config("C4", 0.03))
    assert t.n_rows >= (1 << 20)
    p = ClusterParams.from_options(t, cluster_mask=synth.CONFIG_MASK["C4"])
    narrow = PinnedTable(t, compact=True)
    get_engine(0).run_host(narrow, t, p)
    ocl, onr, _ = orc.oracle_cluster(t, p)
    assert np.array_equal(narrow.out_cluster[:t.n_reads].numpy(), ocl)
    assert np.array_equal(narrow.out_n_reads[:t.n_reads].numpy(), onr)
