"""The reference's tie order on the device file routes: ParsedBed / BamTable.cluster(tie_order="reference"),
cluster_step_fast(tie_order=...), bam_to_clusters and the command line's --tie-order.  The device builds the start column
cluster.py:114 sorts (fslrc_filling_starts), the host sorts it with the reference's own pandas call
(cluster.reference_order_of_starts) and the permutation goes back as the `order` of the clustering call.  Checked against
the reference's stored files without any injected permutation, the host permutation (cluster.reference_tie_order), the
pandas route (pipeline.cluster_step) and, for the command line, the argument routing."""
import ctypes as C
import gzip
import io
import json
import os

import numpy as np
import pandas as pd
import pytest

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
with gzip.open(os.path.join(HERE, "dropin_cases.json.gz")) as _f:
    CASES = json.loads(_f.read())
IDS = [c["name"] for c in CASES]
BY_NAME = {c["name"]: c for c in CASES}
HEADER = b"chrom\trstart\trend\tqname\tn_alignments\taln_size\tqstart\tqend\talignment_score\n"


def _raw(df):
    return df.to_csv(index=False, sep="\t").encode()


def _opts(case):
    return {k: v for k, v in case["opts"].items() if k != "filter_false"}


def _parse(case):
    """The case's UNFILTERED rows parsed on the device, filtered there when the case says so; no permutation injected."""
    from fslr_b200 import tsv
    return tsv.read_mappings_bed(_raw(pd.DataFrame(case["rows"], columns=case["columns"])), dict(case["chr_lengths"]),
                                 filter_false=case["opts"].get("filter_false", False))


def _host_starts(df):
    """The `start` column of the fillings frame keep_fillings makes of df (cluster.py:14-31,111), computed with pandas."""
    rid = pd.factorize(df["qname"])[0]
    idx = pd.Series(np.arange(len(rid)))
    g = idx.groupby(rid)
    keep = ((idx != g.transform("min")) & (idx != g.transform("max"))).to_numpy()
    return np.minimum(df["rstart"].to_numpy(), df["rend"].to_numpy())[keep]


def _host_order(df, lengths, filter_false):
    from fslr_b200 import cluster
    from fslr_b200.table import ColumnarTable
    if filter_false:
        df = cluster.delete_false(df)
    return cluster.reference_tie_order(ColumnarTable.from_dataframe(df, lengths))


def _cluster_bed(case, tie_order):
    pb = _parse(case)
    try:
        pb.cluster(tie_order=tie_order, **_opts(case))
        return pb.cluster_bed_bytes().tobytes()
    finally:
        pb.close()


def _c3_shuffled(filter_false, scale=0.02, seed=3):
    """C3 with its rows shuffled (the rows of a read are no longer contiguous); with filter_false ~20 % of the reads get a
    name containing "False"."""
    from fslr_b200 import synth
    t = synth.make_config("C3", scale)
    df = t.to_dataframe().sample(frac=1.0, random_state=seed).reset_index(drop=True)
    if filter_false:
        rid = pd.factorize(df["qname"])[0]
        hit = np.random.default_rng(seed).random(rid.max() + 1) < 0.2
        df["qname"] = np.where(hit[rid], df["qname"] + "_False", df["qname"])
    raw = _raw(df)
    return raw, pd.read_csv(io.BytesIO(raw), sep="\t"), t.chr_lengths


def test_the_stored_cases_cover_ties_and_early_returns():
    assert len(CASES) == 44
    assert {c["name"] for c in CASES if c["expected"]["cluster_bed"] is None} == {"F6_noclusters", "rand03"}


def test_reference_order_of_starts_is_the_stored_permutation():
    """No GPU: the host half of reference mode, fed the start column of every stored case (as int32, the device's dtype:
    it is sorted as int64 all the same).  34 of the 44 permutations are not the stable one."""
    from fslr_b200 import cluster
    n_unstable = 0
    for case in CASES:
        df = pd.DataFrame(case["rows"], columns=case["columns"])
        if case["opts"].get("filter_false"):
            df = cluster.delete_false(df)
        start = _host_starts(df)
        got = cluster.reference_order_of_starts(start.astype(np.int32))
        assert got.dtype == np.int32 and got.tolist() == case["expected"]["order"], case["name"]
        n_unstable += got.tolist() != np.argsort(start, kind="stable").tolist()
    assert n_unstable == 34


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_stored_files_with_the_reference_tie_order(case):
    """The main check: with tie_order="reference" and nothing injected, both rendered files are the reference's own."""
    exp = case["expected"]
    pb = _parse(case)
    try:
        assert pb.order is None
        res = pb.cluster(tie_order="reference", **_opts(case))
        if exp["cluster_bed"] is None:
            assert res.no_clusters
            return
        assert not res.no_clusters
        assert pb.cluster_bed_bytes().tobytes() == exp["cluster_bed"].encode()
        assert pb.representative_bed_bytes().tobytes() == exp["representative_bed"].encode()
    finally:
        pb.close()


@pytest.mark.gpu
def test_ties_decide_the_numbering():
    """F3_ties: the stable order numbers the clusters differently, so the stored-file check above has teeth."""
    case = BY_NAME["F3_ties"]
    assert _cluster_bed(case, "reference") == case["expected"]["cluster_bed"].encode()
    assert _cluster_bed(case, "stable") != case["expected"]["cluster_bed"].encode()


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_device_permutation_of_the_stored_cases(case):
    df = pd.DataFrame(case["rows"], columns=case["columns"])
    host = _host_order(df, dict(case["chr_lengths"]), case["opts"].get("filter_false", False))
    pb = _parse(case)
    try:
        got = pb.engine.reference_order(pb)
        assert got.device == pb.engine.device and str(got.dtype) == "torch.int32"
        assert got.cpu().numpy().tolist() == host.tolist() == case["expected"]["order"]
    finally:
        pb.close()


@pytest.mark.gpu
@pytest.mark.parametrize("filter_false", [False, True])
def test_device_permutation_with_reads_apart(filter_false):
    from fslr_b200 import tsv
    raw, df, lens = _c3_shuffled(filter_false)
    rid = pd.factorize(df["qname"])[0]
    assert (np.diff(rid) != 0).sum() > 2 * (rid.max() + 1)                  # the rows of most reads are apart
    host = _host_order(df, lens, filter_false)
    from fslr_b200 import cluster
    want = _host_starts(cluster.delete_false(df) if filter_false else df)
    pb = tsv.read_mappings_bed(raw, lens, filter_false=filter_false)
    try:
        assert (pb.n_rows < len(df)) == filter_false
        starts = pb.engine.filling_starts(pb).cpu().numpy()
        assert np.array_equal(starts, want)
        assert len(np.unique(starts)) < len(starts)                          # the table has ties
        assert np.array_equal(pb.engine.reference_order(pb).cpu().numpy(), host)
    finally:
        pb.close()


@pytest.mark.gpu
def test_pipeline_on_a_table_with_ties(tmp_path):
    """C2 at full size (100k reads): the device route in reference mode writes the pandas route's files byte for byte."""
    from fslr_b200 import pipeline, synth
    t = synth.make_config("C2", 1.0)
    raw = _raw(t.to_dataframe())
    df, lens, mask = pd.read_csv(io.BytesIO(raw), sep="\t"), t.chr_lengths, synth.CONFIG_MASK["C2"]
    dev, stable, ref = str(tmp_path / "dev"), str(tmp_path / "stable"), str(tmp_path / "ref")
    assert pipeline.cluster_step_fast(raw, lens, dev, cluster_mask=mask, tie_order="reference") is not None
    assert pipeline.cluster_step_fast(raw, lens, stable, cluster_mask=mask, tie_order="stable") is not None
    assert pipeline.cluster_step(df, lens, cluster_mask=mask, tie_order="reference", out_base=ref) is not None
    for f in (".mappings.cluster.bed", ".mappings.representative.bed"):
        assert open(dev + f, "rb").read() == open(ref + f, "rb").read(), f
    a = pd.read_csv(dev + ".mappings.cluster.bed", sep="\t").groupby("qname", sort=False)["cluster"].first()
    b = pd.read_csv(stable + ".mappings.cluster.bed", sep="\t").groupby("qname", sort=False)["cluster"].first()
    assert 0 < int((a.fillna(-1) != b.fillna(-1)).sum())


@pytest.mark.gpu
def test_bam_route(tmp_path):
    from fslr_b200 import cluster, pipeline, synth_bam as sb
    refs, recs, primers = sb.make_alignments(1500, seed=44, refs=[("chr1", 6000), ("chr2", 5000)], p_single=0.1)
    bam = str(tmp_path / "t.bam")
    sb.write_bam(bam, refs, [sb.encode_record(*r) for r in recs])
    dev, ref = str(tmp_path / "d"), str(tmp_path / "r")
    assert pipeline.bam_to_clusters(bam, primers, dev, fslr_version="9.9", cluster_mask="", tie_order="reference") is not None
    df = pd.read_csv(dev + ".mappings.bed", sep="\t")
    assert pipeline.cluster_step(df, cluster.get_chromosome_lengths(bam), cluster_mask="", tie_order="reference",
                                 out_base=ref) is not None
    for s in (".mappings.cluster.bed", ".mappings.representative.bed"):
        assert open(dev + s, "rb").read() == open(ref + s, "rb").read(), s


def _rows(reads):
    """A small mappings table: reads = [(qname, [(chrom, rstart, rend), ...]), ...]; every row spans 100 query bases."""
    lines = [HEADER]
    for q, rows in reads:
        for k, (c, s, e) in enumerate(rows):
            lines.append(("%s\t%d\t%d\t%s\t%d\t100\t%d\t%d\t60\n" % (c, s, e, q, len(rows), 100 * k, 100 * k + 100)).encode())
    return b"".join(lines)


@pytest.mark.gpu
def test_no_fillings_header_only_and_one_read(tmp_path):
    from fslr_b200 import pipeline, tsv
    lens = {"chr1": 100000}
    raw = _rows([("a", [("chr1", 10, 110)]), ("b", [("chr1", 500, 600), ("chr1", 900, 1000)]), ("c", [("chr1", 10, 110)])])
    pb = tsv.read_mappings_bed(raw, lens)
    try:
        assert pb.engine.filling_starts(pb).numel() == 0
        assert pb.engine.reference_order(pb).numel() == 0
        assert pb.cluster(cluster_mask="", tie_order="reference").no_clusters
    finally:
        pb.close()
    assert pipeline.cluster_step_fast(HEADER, {}, str(tmp_path / "h"), tie_order="reference") is None
    one = _rows([("a", [("chr1", 5000, 5100), ("chr1", 300, 200), ("chr1", 300, 400), ("chr1", 100, 300), ("chr1", 900, 950)])])
    pb = tsv.read_mappings_bed(one, lens)
    try:
        assert pb.engine.filling_starts(pb).cpu().tolist() == [200, 300, 100]
        assert pb.engine.reference_order(pb).cpu().tolist() == [2, 0, 1]
        assert pb.cluster(cluster_mask="", tie_order="reference").no_clusters
    finally:
        pb.close()


@pytest.mark.gpu
def test_modes_alternate_on_one_table():
    """reference, stable, reference on one ParsedBed: each call equals a fresh table clustered in that mode (the cached
    reference order is not left on the table for the stable call)."""
    case = BY_NAME["F3_ties"]
    fresh = {m: _cluster_bed(case, m) for m in ("reference", "stable")}
    assert fresh["reference"] != fresh["stable"]
    pb = _parse(case)
    try:
        for m in ("reference", "stable", "reference", None):
            pb.cluster(tie_order=m, **_opts(case))
            assert pb.cluster_bed_bytes().tobytes() == fresh[m or "stable"], m
        assert pb.order is None
        with pytest.raises(ValueError):
            pb.cluster(tie_order="unstable")
    finally:
        pb.close()


@pytest.mark.gpu
def test_filling_starts_errors():
    import torch
    from fslr_b200 import cluster, synth
    from fslr_b200.engine import DeviceTable, get_engine
    eng = get_engine(0)
    t = synth.make_config("C1", 0.01)
    dtab = DeviceTable(t, eng.device)
    out = torch.empty(t.n_rows, dtype=torch.int32, device=eng.device)
    n = C.c_int64()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(tab, ptr=out.data_ptr(), cap=t.n_rows, nptr=C.byref(n)):
        return eng.lib.fslrc_filling_starts(eng.ctx, C.byref(tab), ptr, cap, nptr, stream)
    assert call(eng._table(dtab, None)) == 0 and n.value == len(cluster.reference_tie_order(t)) > 0
    assert call(eng._table(dtab, None), cap=t.n_rows - 1) == -2
    assert call(eng._table(dtab, None), ptr=None) == -2
    assert call(eng._table(dtab, None), nptr=None) == -2
    assert eng.lib.fslrc_filling_starts(eng.ctx, None, out.data_ptr(), t.n_rows, C.byref(n), stream) == -2
    wire = eng._table(dtab, None)
    wire.read_id = None
    assert call(wire) == -2
    short = eng._table(dtab, None)
    short.n_reads = int(t.read_id.max())                                  # the last read id is out of range
    assert call(short) == -7
    assert call(eng._table(dtab, None)) == 0                               # the context is usable after the errors


def test_cli_passes_tie_order_to_every_route(tmp_path, monkeypatch):
    """No GPU: --tie-order reaches cluster_step_fast (--fast-io), bam_to_clusters (--bam) and cluster_step; unset, each route
    is called exactly as before (no tie_order argument: its own default)."""
    from fslr_b200 import pipeline
    calls = []
    monkeypatch.setattr(pipeline, "bam_to_clusters", lambda *a, **k: calls.append(("bam", a, k)))
    monkeypatch.setattr(pipeline, "cluster_step_fast", lambda *a, **k: calls.append(("fast", a, k)))
    monkeypatch.setattr(pipeline, "cluster_step", lambda *a, **k: calls.append(("pandas", a, k)))
    lens = tmp_path / "lens.json"
    lens.write_text('{"chr1": 1000}')
    pcsv = tmp_path / "primers.csv"
    pcsv.write_text("primer_name,primer_seq\n21q1,ACGT\n")
    bed = ["--bed", "x.bed", "--chr-lengths", str(lens), "--out-base", "o"]
    bam = ["--bam", "x.bam", "--primers-csv", str(pcsv), "--primers", "21q1", "--out-base", "o"]
    for tie in (["--tie-order", "reference"], ["--tie-order", "stable"], []):
        pipeline.main(bed + ["--fast-io"] + tie)
        pipeline.main(bam + tie)
        pipeline.main(bed + tie)
    assert [c[0] for c in calls] == ["fast", "bam", "pandas"] * 3
    assert [c[2].get("tie_order") for c in calls] == ["reference"] * 3 + ["stable"] * 3 + [None] * 3
    assert all("tie_order" not in c[2] for c in calls[6:])
    with pytest.raises(SystemExit):
        pipeline.main(bed + ["--tie-order", "unstable"])
