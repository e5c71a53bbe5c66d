"""--filter-false on the device file path (fslrc_tsv_delete_false, read_mappings_bed(filter_false=True)): the reads whose qname
contains "False" leave the parsed table before the clustering, as main.py:229-230 drops them with cluster.delete_false.
Checked against the reference's stored files, the pandas route (pipeline.cluster_step) and, for the command line, the
argument routing."""
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
    _ALL = json.loads(_f.read())
FILTERED = [c for c in _ALL if c["opts"].get("filter_false")]
KEPT = [c for c in _ALL if not c["opts"].get("filter_false") and any("False" in str(r[c["columns"].index("qname")]) for r in c["rows"])]
NUMERIC = ("rstart", "rend", "aln_size", "qstart", "qend", "n_alignments", "alignment_score")


def _raw(df):
    return df.to_csv(index=False, sep="\t").encode()


def _stored_case(case, filter_false):
    """The case's UNFILTERED rows parsed on the device (filtered there or not), the reference's tie permutation injected,
    clustered with the case's options; both rendered files against the reference's own."""
    import torch
    from fslr_b200 import tsv
    exp = case["expected"]
    pb = tsv.read_mappings_bed(_raw(pd.DataFrame(case["rows"], columns=case["columns"])), dict(case["chr_lengths"]),
                               filter_false=filter_false)
    try:
        pb.order = torch.tensor(exp["order"], dtype=torch.int32, device=pb.engine.device)
        res = pb.cluster(**{k: v for k, v in case["opts"].items() if k != "filter_false"})
        if exp["cluster_bed"] is None:
            assert res.no_clusters
            return res
        assert not res.no_clusters
        assert pb.cluster_bed_bytes().tobytes() == exp["cluster_bed"].encode()
        assert pb.representative_bed_bytes().tobytes() == exp["representative_bed"].encode()
        return res
    finally:
        pb.close()


def test_the_stored_cases_cover_both_sides():
    assert len(FILTERED) == 11 and len(KEPT) == 7
    assert {"F6_false_filtered", "F6_false_kept", "rand03"} <= {c["name"] for c in FILTERED + KEPT}


@pytest.mark.gpu
@pytest.mark.parametrize("case", FILTERED, ids=[c["name"] for c in FILTERED])
def test_stored_filtered_cases(case):
    _stored_case(case, True)


@pytest.mark.gpu
@pytest.mark.parametrize("case", KEPT, ids=[c["name"] for c in KEPT])
def test_stored_cases_with_false_names_and_no_filter(case):
    res = _stored_case(case, False)
    if case["name"] == "rand03":
        assert res.no_clusters


def _synth_frame(scale=0.02, seed=5):
    """C3 with ~20 % of the reads renamed so that their names contain "False" (prefix, suffix, middle, the whole name for
    one read) and ~8 % carrying near misses that must be kept."""
    from fslr_b200 import synth
    t = synth.make_config("C3", scale)
    df = t.to_dataframe()
    names = t.qnames()
    rng = np.random.default_rng(seed)
    u = rng.random(t.n_reads)
    kind = rng.integers(0, 4, t.n_reads)
    miss = ("false", "FALSE", "Fals", "Fa_lse")
    new = []
    first = np.unique(t.read_id, return_index=True)[1]                   # first row of every read id
    for r, q in enumerate(names[first].tolist()):
        if u[r] < 0.2:
            q = ("False" + q, q + "_False", q[:8] + "False" + q[8:], q + ".False_False")[kind[r]]
        elif u[r] < 0.28:
            q = q[:8] + miss[kind[r]] + q[8:]
        new.append(q)
    whole = int(np.flatnonzero(u >= 0.28)[0])
    new[whole] = "False"
    df["qname"] = np.array(new, dtype=object)[t.read_id]
    raw = _raw(df)
    return raw, pd.read_csv(io.BytesIO(raw), sep="\t"), t.chr_lengths


@pytest.mark.gpu
def test_synthetic_files_equal_the_pandas_route(tmp_path):
    from fslr_b200 import pipeline, synth
    raw, df, lens = _synth_frame()
    assert 0.15 < df["qname"].drop_duplicates().str.contains("False").mean() < 0.25
    mask = synth.CONFIG_MASK["C3"]
    dev, ref = str(tmp_path / "dev"), str(tmp_path / "ref")
    assert pipeline.cluster_step_fast(raw, lens, dev, cluster_mask=mask, filter_false=True) is not None
    assert pipeline.cluster_step(df, lens, cluster_mask=mask, filter_false=True, tie_order="stable", out_base=ref) is not None
    for f in (".mappings.cluster.bed", ".mappings.representative.bed"):
        assert open(dev + f, "rb").read() == open(ref + f, "rb").read(), f


@pytest.mark.gpu
def test_synthetic_parsed_columns_equal_the_filtered_frame():
    from fslr_b200 import cluster, tsv
    from fslr_b200.table import ColumnarTable
    raw, df, lens = _synth_frame()
    filtered = cluster.delete_false(df)
    ref = ColumnarTable.from_dataframe(filtered, lens)
    pb = tsv.read_mappings_bed(raw, lens, filter_false=True)
    try:
        assert (pb.n_rows, pb.n_reads) == (ref.n_rows, ref.n_reads) == (len(filtered), filtered["qname"].nunique())
        assert pb.n_rows < len(df)
        assert np.array_equal(pb.column("read_id"), ref.read_id)
        assert list(pb.qnames()) == list(ref.qnames)
        assert pb.chrom_names == [str(c) for c in pd.factorize(df["chrom"])[1]]          # the unfiltered numbering
        assert np.array_equal(np.array(pb.chrom_names, dtype=object)[pb.column("chrom")],
                              np.array(ref.chrom_names, dtype=object)[ref.chrom])
        for k in NUMERIC:
            assert np.array_equal(pb.column(k), filtered[k].to_numpy()), k
        assert pb.filter_ms > 0
    finally:
        pb.close()


def _small(tmp_rename):
    from fslr_b200 import synth
    t = synth.make_config("C1", 0.05)
    df = t.to_dataframe()
    df["qname"] = [tmp_rename(q) for q in df["qname"]]
    return _raw(df), t.chr_lengths


@pytest.mark.gpu
def test_every_read_filtered(tmp_path):
    from fslr_b200 import pipeline, tsv
    raw, lens = _small(lambda q: q + "False")
    pb = tsv.read_mappings_bed(raw, lens, filter_false=True)
    assert (pb.n_rows, pb.n_reads) == (0, 0)
    assert pb.cluster_bed_bytes().tobytes() == raw[:raw.index(b"\n")] + b"\tcluster\tn_reads\n"
    pb.close()
    base = str(tmp_path / "o")
    assert pipeline.cluster_step_fast(raw, lens, base, filter_false=True) is None
    assert pipeline.cluster_step(pd.read_csv(io.BytesIO(raw), sep="\t"), lens, filter_false=True, out_base=base) is None
    assert not os.path.exists(base + ".mappings.cluster.bed") and not os.path.exists(base + ".mappings.representative.bed")


@pytest.mark.gpu
def test_no_read_filtered_is_byte_identical(tmp_path):
    from fslr_b200 import pipeline
    raw, lens = _small(lambda q: q + ".false_FALSE")                     # near misses only
    out = {}
    for ff in (False, True):
        base = str(tmp_path / str(ff))
        assert pipeline.cluster_step_fast(raw, lens, base, filter_false=ff) is not None
        out[ff] = [open(base + f, "rb").read() for f in (".mappings.cluster.bed", ".mappings.representative.bed")]
    assert out[True] == out[False]


@pytest.mark.gpu
def test_header_only(tmp_path):
    from fslr_b200 import pipeline, tsv
    raw = b"chrom\trstart\trend\tqname\tn_alignments\taln_size\tqstart\tqend\talignment_score\n"
    pb = tsv.read_mappings_bed(raw, {}, filter_false=True)
    assert (pb.n_rows, pb.n_reads) == (0, 0)
    pb.close()
    assert pipeline.cluster_step_fast(raw, {}, str(tmp_path / "o"), filter_false=True) is None


@pytest.mark.gpu
def test_malformed_rows_of_dropped_reads_still_raise():
    from fslr_b200 import tsv
    from fslr_b200._native import FslrError
    raw, lens = _small(lambda q: q)
    lines = raw.split(b"\n")
    f = lines[5].split(b"\t")
    f[3] = b"x_False_" + f[3]
    bad_int = list(f); bad_int[1] = b"12x4"
    for bad in (b"\t".join(bad_int), b"\t".join(f[:3])):
        with pytest.raises(FslrError):
            tsv.read_mappings_bed(b"\n".join(lines[:5] + [bad] + lines[5:]), lens, filter_false=True)
    pb = tsv.read_mappings_bed(b"\n".join(lines[:5] + [b"\t".join(f)] + lines[5:]), lens, filter_false=True)
    assert pb.n_rows == len(lines) - 2
    pb.close()


@pytest.mark.gpu
def test_a_second_call_removes_nothing():
    import torch
    from fslr_b200 import _native, tsv
    from fslr_b200.engine import get_engine
    raw, df, lens = _synth_frame(0.005, seed=9)
    pb = tsv.read_mappings_bed(raw, lens, filter_false=True)
    try:
        before = {k: pb.column(k) for k in ("read_id", "chrom") + NUMERIC}
        names = list(pb.qnames())
        pb.cluster()
        bed = pb.cluster_bed_bytes().tobytes()
        info = _native.TsvInfo.from_buffer_copy(pb.info)
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        pb.engine._check(pb.engine.lib.fslrc_tsv_delete_false(pb.engine.ctx, C.byref(info), stream))
        assert (info.n_rows, info.n_reads, info.read_id, info.rstart) == (pb.n_rows, pb.n_reads, pb.info.read_id, pb.info.rstart)
        assert all(np.array_equal(pb.column(k), v) for k, v in before.items())
        pb._names = None
        assert list(pb.qnames()) == names
        assert pb.cluster_bed_bytes().tobytes() == bed
    finally:
        pb.close()
    eng = get_engine(0)                                                 # no open table
    info = _native.TsvInfo()
    assert eng.lib.fslrc_tsv_delete_false(eng.ctx, C.byref(info), C.c_void_p(torch.cuda.current_stream().cuda_stream)) == -2


@pytest.mark.gpu
def test_bam_route(tmp_path):
    from fslr_b200 import cluster, pipeline, synth_bam as sb
    refs, recs, primers = sb.make_alignments(1500, seed=43, refs=[("chr1", 6000), ("chr2", 5000)], p_single=0.1)
    bam = str(tmp_path / "t.bam")
    sb.write_bam(bam, refs, [sb.encode_record(*r) for r in recs])
    f, u, ref = str(tmp_path / "f"), str(tmp_path / "u"), str(tmp_path / "r")
    assert pipeline.bam_to_clusters(bam, primers, f, fslr_version="9.9", cluster_mask="", filter_false=True) is not None
    assert pipeline.bam_to_clusters(bam, primers, u, fslr_version="9.9", cluster_mask="") is not None
    bed = open(f + ".mappings.bed", "rb").read()
    assert bed == open(u + ".mappings.bed", "rb").read()                # mappings.bed is written before the filter
    df = pd.read_csv(io.BytesIO(bed), sep="\t")
    assert 0 < df["qname"].str.contains("False").sum() < len(df)
    lengths = cluster.get_chromosome_lengths(bam)
    assert pipeline.cluster_step(df, lengths, cluster_mask="", filter_false=True, tie_order="stable", out_base=ref) is not None
    for s in (".mappings.cluster.bed", ".mappings.representative.bed"):
        assert open(f + s, "rb").read() == open(ref + s, "rb").read(), s
    assert open(f + ".mappings.cluster.bed", "rb").read() != open(u + ".mappings.cluster.bed", "rb").read()


def test_cli_passes_filter_false_to_the_device_routes(tmp_path, monkeypatch):
    """No GPU: the command line routes --fast-io --filter-false and --bam --filter-false to the device path with the flag."""
    from fslr_b200 import pipeline
    calls = []
    monkeypatch.setattr(pipeline, "bam_to_clusters", lambda *a, **k: calls.append(("bam", a, k)))
    monkeypatch.setattr(pipeline, "cluster_step_fast", lambda *a, **k: calls.append(("fast", a, k)))
    monkeypatch.setattr(pipeline, "cluster_step", lambda *a, **k: calls.append(("pandas", a, k)))
    lens = tmp_path / "lens.json"
    lens.write_text('{"chr1": 1000}')
    pcsv = tmp_path / "primers.csv"
    pcsv.write_text("primer_name,primer_seq\n21q1,ACGT\n")
    pipeline.main(["--bed", "x.bed", "--chr-lengths", str(lens), "--out-base", "o", "--fast-io", "--filter-false"])
    pipeline.main(["--bam", "x.bam", "--primers-csv", str(pcsv), "--primers", "21q1", "--out-base", "o", "--filter-false"])
    pipeline.main(["--bed", "x.bed", "--chr-lengths", str(lens), "--out-base", "o", "--fast-io"])
    assert [c[0] for c in calls] == ["fast", "bam", "fast"]
    assert calls[0][2]["filter_false"] is True and calls[1][2]["filter_false"] is True
    assert calls[2][2]["filter_false"] is False
