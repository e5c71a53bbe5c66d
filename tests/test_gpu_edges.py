"""The similarity graph from the device (fslrc_set_edge_capture / fslrc_edges / fslrc_tsv_write_edges): every edge the
clustering handed to union-find, as (read whose query tested the pair, other read, Jaccard similarity), against the CPU
oracle's literal loop (cluster.py:187-227), on the stored cases, at full size, through every entry and file route."""
import ctypes as C
import gzip
import io
import json
import os

import numpy as np
import pandas as pd
import pytest

from tests import golden_io
from tests.test_oracle_edges import partition_of_edges, same_partition

pytestmark = pytest.mark.gpu

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
with gzip.open(os.path.join(HERE, "dropin_cases.json.gz")) as _f:
    DROPIN = json.loads(_f.read())
HEADER = b"query1\tquery2\tjaccard_similarity\n"


@pytest.fixture(scope="module")
def engine():
    from fslr_b200.engine import get_engine
    return get_engine(0)


def query_rank(t, params, order=None):
    """Per read id the rank at which cluster.py:197 visits it as a query (-1: no interval): order of first appearance in
    the masked, sorted fillings (cluster.py:14-31,89-121,189-191)."""
    rid = np.asarray(t.read_id)
    idx = np.arange(rid.shape[0])
    first = np.full(t.n_reads, rid.shape[0])
    last = np.full(t.n_reads, -1)
    np.minimum.at(first, rid, idx)
    np.maximum.at(last, rid, idx)
    rows = idx[(idx != first[rid]) & (idx != last[rid])]
    s = np.minimum(t.rstart[rows], t.rend[rows]).astype(np.int64)
    e = np.maximum(t.rstart[rows], t.rend[rows]).astype(np.int64)
    o = np.asarray(order, dtype=np.int64) if order is not None else np.argsort(s, kind="stable")
    rows, s, e = rows[o], s[o], e[o]
    ch = np.asarray(t.chrom)[rows]
    drop = np.zeros(len(rows), bool)
    if params.chrom_masked is not None and len(params.chrom_masked):
        drop |= np.asarray(params.chrom_masked, bool)[ch]
    if params.mask_subtelomere:
        cl = np.asarray(t.chrom_len, np.int64)[ch]
        drop |= (cl > 1000000) & ((s < params.subtel) | (cl - e < params.subtel))
    drid = rid[rows][~drop]
    u, fi = np.unique(drid, return_index=True)
    q = np.full(t.n_reads, -1)
    q[u[np.argsort(fi, kind="stable")]] = np.arange(len(u))
    return q


def rows_of(r1, r2, jac):
    return set(zip(np.asarray(r1).tolist(), np.asarray(r2).tolist(), np.asarray(jac, np.float64).view(np.uint64).tolist()))


def check(res, t, params, order=None, oracle=None, name=""):
    """res (a captured ClusterResult) against the oracle: the same directed rows, Jaccard bits included; counts; no pair
    twice; components = the returned partition; rows in query-rank order."""
    from tests.oracle_edges import oracle_cluster_edges
    if oracle is None:
        oracle = oracle_cluster_edges(t, params, order=order)
    ocl, onr, ost, (o1, o2, oj) = oracle
    e = res.edges
    assert e.read1.dtype == np.int32 and e.read2.dtype == np.int32 and e.jaccard.dtype == np.float64, name
    assert len(e.read1) == res.stats["edges"] == ost["edges"], name
    assert rows_of(e.read1, e.read2, e.jaccard) == rows_of(o1, o2, oj), name
    lo, hi = np.minimum(e.read1, e.read2), np.maximum(e.read1, e.read2)
    assert len(set(zip(lo.tolist(), hi.tolist()))) == len(lo), name
    assert np.array_equal(res.cluster, ocl) and np.array_equal(res.n_reads, onr), name
    assert same_partition(partition_of_edges(t.n_reads, e.read1, e.read2), res.cluster, res.n_reads), name
    q = query_rank(t, params, order).astype(np.int64)
    key = q[e.read1] * (int(q.max()) + 2) + q[e.read2]
    assert np.all(np.diff(key) > 0), name
    return oracle


# ---------------------------------------------------------------- stored cases
@pytest.mark.parametrize("fname,n", [("small_cases.npz", 415), ("wide_cases.npz", 120), ("config_cases.npz", 8)])
def test_stored_cases(engine, fname, n):
    cases = golden_io.load(fname)
    assert len(cases) == n
    bad = []
    for c in cases:
        try:
            check(engine.cluster(c.table, c.params, order=c.order, edges=True), c.table, c.params, c.order, name=c.name)
        except AssertionError as ex:
            bad.append(str(ex) or c.name)
    assert not bad, "%d/%d cases differ: %s" % (len(bad), n, bad[:5])


def _dropin_table(case):
    from fslr_b200 import cluster
    from fslr_b200.table import ClusterParams, ColumnarTable
    df = pd.DataFrame(case["rows"], columns=case["columns"])
    if case["opts"].get("filter_false"):
        df = cluster.delete_false(df)
    t = ColumnarTable.from_dataframe(df, dict(case["chr_lengths"]))
    p = ClusterParams.from_options(t, **{k: v for k, v in case["opts"].items() if k != "filter_false"})
    return t, p, np.asarray(case["expected"]["order"], dtype=np.int64)


def test_dropin_tables(engine):
    assert len(DROPIN) == 44
    for case in DROPIN:
        t, p, order = _dropin_table(case)
        check(engine.cluster(t, p, order=order, edges=True), t, p, order, name=case["name"])


def _drop_in_block(case, **kw):
    """main.py:211-242 with fslr_b200.cluster (as tests/test_gpu_dropin.py runs it)."""
    from fslr_b200 import cluster
    o = case["opts"]
    bed = pd.DataFrame(case["rows"], columns=case["columns"])
    mask = set()
    cm = o.get("cluster_mask", "subtelomere")
    if cm:
        allowed = set(bed["chrom"])
        mask = {i for i in cm.split(",") if i in allowed or i == "subtelomere"}
    cutoffs = [float(i) for i in o.get("jaccard_cutoffs", "1,1,0.66,0.66,0.66,0.5").split(",")]
    bed, lens, mask, _ = cluster.rename_chromosomes(bed, dict(case["chr_lengths"]), mask)
    if o.get("filter_false"):
        bed = cluster.delete_false(bed)
    data = cluster.prepare_data(cluster.keep_fillings(bed), mask, lens, threshold=500_000)
    return cluster.query_interval_trees(cluster.build_interval_trees(data), data, o.get("overlap", 0.8), cutoffs,
                                        o.get("edge_threshold", 10), o.get("qlen_diff", 0.04), o.get("n_alignment_diff", 0.25), **kw)


def test_query_interval_trees_with_matches():
    from tests.oracle_edges import oracle_cluster_edges
    for case in DROPIN:
        t, p, order = _dropin_table(case)
        _, _, _, (o1, o2, oj) = oracle_cluster_edges(t, p, order=order)
        q = np.asarray(t.qnames, dtype=object)
        want = set(zip(q[o1].tolist(), q[o2].tolist(), oj.view(np.uint64).tolist()))
        match_df, G = _drop_in_block(case, with_matches=True)
        assert list(match_df.columns) == ["query1", "query2", "jaccard_similarity"], case["name"]
        got = set(zip(match_df["query1"].tolist(), match_df["query2"].tolist(),
                      match_df["jaccard_similarity"].to_numpy(np.float64).view(np.uint64).tolist()))
        assert got == want and len(match_df) == len(want) == G.number_of_edges(), case["name"]
        assert G.edges() == list(zip(match_df["query1"], match_df["query2"])), case["name"]
        empty, G0 = _drop_in_block(case)
        assert empty.empty and list(empty.columns) == ["query1", "query2", "jaccard_similarity"]
        with pytest.raises(RuntimeError):
            G0.edges()


# ---------------------------------------------------------------- full size
@pytest.mark.parametrize("name", ["C1", "C2", "C3", "C5"])
def test_fullsize_entries(engine, name, monkeypatch):
    """The host and the device entry, wide and wire-format columns, the fast and the general ingest: one oracle run."""
    import torch
    from fslr_b200 import synth
    from fslr_b200.engine import ClusterResult, DeviceTable, PinnedTable
    from fslr_b200.table import ClusterParams, ColumnarTable
    t = ColumnarTable.from_synth(synth.make_config(name))
    p = ClusterParams.from_options(t, cluster_mask=synth.CONFIG_MASK[name])
    ora = check(engine.cluster(t, p, edges=True), t, p, name=name)                        # host entry, fast ingest
    ptab = PinnedTable(t, compact=True)
    st = engine.run_host(ptab, t, p, edges=True)
    n = t.n_reads
    check(ClusterResult(ptab.out_cluster[:n].numpy().copy(), ptab.out_n_reads[:n].numpy().copy(), False, st,
                        engine.edge_list()), t, p, oracle=ora, name=name + " wire")
    d = DeviceTable(t, engine.device)
    st, el = engine.run_resident(d, t, p, edges=True)
    torch.cuda.synchronize()
    check(ClusterResult(d.out_cluster[:n].cpu().numpy(), d.out_n_reads[:n].cpu().numpy(), False, st, el), t, p, oracle=ora,
          name=name + " device")
    if name == "C3":
        monkeypatch.setenv("FSLRC_GENERAL_INGEST", "1")
        check(engine.cluster(t, p, edges=True), t, p, oracle=ora, name=name + " general ingest")


def test_tie_orders_give_their_own_edges(engine):
    """C2 (duplicate families with equal starts): the reference tie order and the stable one each match the oracle run
    with the same order; the edge sets differ."""
    from fslr_b200 import cluster, synth
    from fslr_b200.table import ClusterParams, ColumnarTable
    t = ColumnarTable.from_synth(synth.make_config("C2"))
    p = ClusterParams.from_options(t, cluster_mask=synth.CONFIG_MASK["C2"])
    order = cluster.reference_tie_order(t)
    ref = engine.cluster(t, p, order=order, edges=True)
    check(ref, t, p, order=order.astype(np.int64), name="reference")
    stable = engine.cluster(t, p, edges=True)
    check(stable, t, p, name="stable")
    assert rows_of(ref.edges.read1, ref.edges.read2, ref.edges.jaccard) != rows_of(stable.edges.read1, stable.edges.read2,
                                                                                    stable.edges.jaccard)


def test_c5_capture_is_repeatable(engine):
    from fslr_b200 import synth
    from fslr_b200.table import ClusterParams, ColumnarTable
    t = ColumnarTable.from_synth(synth.make_config("C5"))
    p = ClusterParams.from_options(t, cluster_mask=synth.CONFIG_MASK["C5"])
    a = engine.cluster(t, p, edges=True)
    assert a.stats["saturating_reads"] > 500000
    b = engine.cluster(t, p, edges=True)
    for k in ("read1", "read2", "jaccard"):
        assert np.array_equal(getattr(a.edges, k), getattr(b.edges, k)), k
    q = query_rank(t, p).astype(np.int64)
    assert np.all(np.diff(q[a.edges.read1] * (int(q.max()) + 2) + q[a.edges.read2]) > 0)


def test_capture_leaves_the_default_path_alone(engine):
    import torch
    from fslr_b200 import synth
    from fslr_b200.engine import DeviceTable, Engine
    from fslr_b200.table import ClusterParams, ColumnarTable
    eng = Engine(0)                                   # a context whose switch was never touched
    t = ColumnarTable.from_synth(synth.make_config("C2", 0.2))
    p = ClusterParams.from_options(t, cluster_mask=synth.CONFIG_MASK["C2"])
    d = DeviceTable(t, eng.device)

    def step(edges):
        n0 = eng.launch_count()
        out = eng.run_resident(d, t, p, edges=edges)
        torch.cuda.synchronize()
        return eng.launch_count() - n0, d.out_cluster.cpu().numpy().copy(), d.out_n_reads.cpu().numpy().copy(), out
    k0, c0, n0, _ = step(False)
    k1, c1, n1, (st, el) = step(True)
    k2, c2, n2, _ = step(False)
    assert k1 > k0 == k2
    assert np.array_equal(c0, c1) and np.array_equal(c0, c2) and np.array_equal(n0, n1) and np.array_equal(n0, n2)
    assert st["edges"] == len(el.read1) > 0
    assert eng.lib.fslrc_edges(eng.ctx, None, None, None, 0, C.byref(C.c_int64()), None) == -2   # switched off: freed
    eng.close()


# ---------------------------------------------------------------- file routes
def _raw(df):
    return df.to_csv(index=False, sep="\t").encode()


def test_edges_bytes_of_the_dropin_tables():
    """The device renderer equals pandas' to_csv of the same rows (qname slicing, repr), filtered tables included."""
    from fslr_b200 import cluster, tsv
    for case in DROPIN:
        o = case["opts"]
        pb = tsv.read_mappings_bed(_raw(pd.DataFrame(case["rows"], columns=case["columns"])), dict(case["chr_lengths"]),
                                   filter_false=o.get("filter_false", False))
        try:
            res = pb.cluster(tie_order="reference", edges=True, **{k: v for k, v in o.items() if k != "filter_false"})
            t, p, order = _dropin_table(case)
            check(res, t, p, order, name=case["name"])
            want = cluster.match_frame(pb.qnames(), res.edges).to_csv(sep="\t", index=False).encode()
            assert pb.edges_bytes().tobytes() == want, case["name"]
        finally:
            pb.close()


def test_fast_io_writes_the_pandas_routes_edges(tmp_path):
    from fslr_b200 import pipeline, synth
    t = synth.make_config("C2", 1.0)
    raw = _raw(t.to_dataframe())
    df, lens, mask = pd.read_csv(io.BytesIO(raw), sep="\t"), t.chr_lengths, synth.CONFIG_MASK["C2"]
    dev, ref = str(tmp_path / "dev.tsv"), str(tmp_path / "ref.tsv")
    assert pipeline.cluster_step_fast(raw, lens, str(tmp_path / "d"), cluster_mask=mask, tie_order="reference", edges=dev) is not None
    assert pipeline.cluster_step(df, lens, cluster_mask=mask, tie_order="reference", out_base=str(tmp_path / "r"), edges=ref) is not None
    a = open(dev, "rb").read()
    assert a == open(ref, "rb").read() and a.count(b"\n") > 1000


def test_filter_false_route(tmp_path):
    """C3 with 20 % of the reads named *_False: read ids of the filtered table, device file = pandas route's file."""
    from fslr_b200 import cluster, pipeline, synth
    from fslr_b200.table import ClusterParams, ColumnarTable
    from tests.test_gpu_tie_order import _c3_shuffled
    raw, df, lens = _c3_shuffled(True)
    mask = synth.CONFIG_MASK["C3"]
    dev, ref = str(tmp_path / "dev.tsv"), str(tmp_path / "ref.tsv")
    res = pipeline.cluster_step_fast(raw, lens, str(tmp_path / "d"), cluster_mask=mask, filter_false=True, edges=dev)
    assert res is not None
    t = ColumnarTable.from_dataframe(cluster.delete_false(df), lens)
    p = ClusterParams.from_options(t, cluster_mask=mask)
    check(res, t, p, name="C3 filtered")
    assert pipeline.cluster_step(df, lens, cluster_mask=mask, filter_false=True, tie_order="stable", out_base=str(tmp_path / "r"),
                                 edges=ref) is not None
    assert open(dev, "rb").read() == open(ref, "rb").read()
    assert b"False" not in open(dev, "rb").read()


def test_bam_route(tmp_path):
    from fslr_b200 import cluster, pipeline, synth_bam as sb
    refs, recs, primers = sb.make_alignments(1500, seed=44, refs=[("chr1", 6000), ("chr2", 5000)], p_single=0.1)
    bam = str(tmp_path / "t.bam")
    sb.write_bam(bam, refs, [sb.encode_record(*r) for r in recs])
    dev, ref = str(tmp_path / "d"), str(tmp_path / "r")
    assert pipeline.bam_to_clusters(bam, primers, dev, fslr_version="9.9", cluster_mask="", tie_order="reference",
                                    edges=dev + ".edges") is not None
    df = pd.read_csv(dev + ".mappings.bed", sep="\t")
    assert pipeline.cluster_step(df, cluster.get_chromosome_lengths(bam), cluster_mask="", tie_order="reference",
                                 out_base=ref, edges=ref + ".edges") is not None
    a = open(dev + ".edges", "rb").read()
    assert a == open(ref + ".edges", "rb").read() and a.count(b"\n") > 10


def test_early_return_writes_the_header(tmp_path):
    from fslr_b200 import pipeline
    from tests.test_gpu_tie_order import _rows
    raw = _rows([("a", [("chr1", 10, 110)]), ("b", [("chr1", 500, 600), ("chr1", 900, 1000)])])
    f1, f2 = str(tmp_path / "f.tsv"), str(tmp_path / "p.tsv")
    assert pipeline.cluster_step_fast(raw, {"chr1": 100000}, str(tmp_path / "x"), cluster_mask="", edges=f1) is None
    assert pipeline.cluster_step(pd.read_csv(io.BytesIO(raw), sep="\t"), {"chr1": 100000}, cluster_mask="", edges=f2) is None
    assert open(f1, "rb").read() == open(f2, "rb").read() == HEADER
    assert pd.DataFrame(columns=["query1", "query2", "jaccard_similarity"]).to_csv(sep="\t", index=False).encode() == HEADER


# ---------------------------------------------------------------- errors
def test_errors(engine):
    import torch
    from fslr_b200 import synth, tsv
    from fslr_b200.engine import DeviceTable
    from fslr_b200.table import ClusterParams, ColumnarTable
    lib, ctx = engine.lib, engine.ctx
    n = C.c_int64()

    def edges(cap=0, buf=None):
        b = buf or (None, None, None)
        return lib.fslrc_edges(ctx, b[0], b[1], b[2], cap, C.byref(n), None)
    t = ColumnarTable.from_synth(synth.make_config("C1", 0.05))
    p = ClusterParams.from_options(t)
    engine.cluster(t, p)
    assert edges() == -2                                                  # no capture
    res = engine.cluster(t, p, edges=True)
    assert edges() == 0 and n.value == len(res.edges.read1) > 1            # size query
    k = n.value
    bufs = [torch.empty(k, dtype=dt, device=engine.device) for dt in (torch.int32, torch.int32, torch.float64)]
    ptrs = [b.data_ptr() for b in bufs]
    assert edges(k - 1, ptrs) == -2                                       # cap too small
    assert edges(k, ptrs) == 0
    torch.cuda.synchronize()
    assert np.array_equal(bufs[0].cpu().numpy(), res.edges.read1) and np.array_equal(bufs[2].cpu().numpy(), res.edges.jaccard)
    assert edges(k, [None, ptrs[1], None]) == 0
    bad = ClusterParams.from_options(t)
    t0 = ColumnarTable.from_synth(synth.make_config("C1", 0.05))
    t0.aln_size = np.zeros_like(t0.aln_size)                             # the reference's ZeroDivisionError: the call fails
    with pytest.raises(Exception):
        engine.cluster(t0, bad, edges=True)
    assert edges() == -2                                                  # after a failed call
    engine.cluster(t, p, edges=True)
    d = DeviceTable(t, engine.device)
    engine._set_capture(True)
    engine.run_sharded(d, t, p, 0, 1)                                     # the multi-GPU sequence, one rank
    assert edges() == -2
    # the renderer: only for a clustering of the table open now
    from tests.test_gpu_tie_order import _rows
    raw = _rows([("a", [("chr1", 10, 110), ("chr1", 10, 110), ("chr1", 10, 110)]),
                 ("b", [("chr1", 10, 110), ("chr1", 10, 110), ("chr1", 10, 110)]),
                 ("xFalse", [("chr1", 10, 110), ("chr1", 10, 110), ("chr1", 10, 110)])])
    pb = tsv.read_mappings_bed(raw, {"chr1": 100000}, device=0)
    try:
        with pytest.raises(Exception):
            pb.edges_bytes()                                              # the last capture was not of this table
        r = pb.cluster(cluster_mask="", edges=True)
        assert len(r.edges.read1) == 3 and pb.edges_bytes().tobytes().startswith(HEADER)
        engine.cluster(t, p, edges=True)                                  # a clustering of another table
        with pytest.raises(Exception):
            pb.edges_bytes()
        pb.cluster(cluster_mask="", edges=True)
        info = pb.info
        assert lib.fslrc_tsv_delete_false(ctx, C.byref(info), None) == 0  # the table changed under the capture
        with pytest.raises(Exception):
            pb.edges_bytes()
    finally:
        pb.close()
    pb = tsv.read_mappings_bed(raw, {"chr1": 100000}, device=0)
    try:
        pb.cluster(cluster_mask="", edges=True)
        out = lib.fslrc_tsv_write_edges(ctx, None, 0, C.byref(n), None)
        assert out == 0 and n.value == len(pb.edges_bytes())
        small = engine.pinned_bytes(n.value)
        assert lib.fslrc_tsv_write_edges(ctx, small.data_ptr(), n.value - 1, C.byref(n), None) == -2
    finally:
        pb.close()
    pb = tsv.read_mappings_bed(raw, {"chr1": 100000}, device=0)
    pb.cluster(cluster_mask="", edges=True)
    pb2 = tsv.read_mappings_bed(raw, {"chr1": 100000}, device=0)        # a re-open replaces the table
    try:
        assert lib.fslrc_tsv_write_edges(ctx, None, 0, C.byref(n), None) == -2
    finally:
        pb2.close()
    engine._set_capture(False)
