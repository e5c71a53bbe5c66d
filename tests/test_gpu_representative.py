"""`<base>.mappings.representative.bed` rendered on the device (ParsedBed.representative_bed_bytes,
fslrc_tsv_write_representative_bed) against the reference's files and against the pandas route it replaces in
pipeline.cluster_step_fast: pd.read_csv of the written cluster.bed, cluster.choose_alignment, DataFrame.to_csv."""
import ctypes as C
import gzip
import io
import json
import os

import numpy as np
import pandas as pd
import pytest
import torch

pytestmark = pytest.mark.gpu

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
with gzip.open(os.path.join(HERE, "dropin_cases.json.gz")) as _f:
    CASES = [c for c in json.loads(_f.read()) if c["expected"]["representative_bed"] is not None]
HEADER = "chrom\trstart\trend\tqname\tn_alignments\taln_size\tqstart\tqend\talignment_score"


def _parse_with_clusters(raw, cluster_of, n_reads_of):
    """Parse `raw` on the device and upload per-read cluster / n_reads ({qname: value}) in place of a clustering run."""
    from fslr_b200 import tsv
    pb = tsv.read_mappings_bed(raw, {})
    names = pb.qnames()
    n = pb.n_reads
    pb.out_cluster[:n].copy_(torch.as_tensor(np.array([cluster_of[q] for q in names], dtype=np.int32)))
    pb.out_n_reads[:n].copy_(torch.as_tensor(np.array([n_reads_of[q] for q in names], dtype=np.int32)))
    return pb


def _pandas_route(cluster_bed):
    """What cluster_step_fast wrote before: the representative file derived from the cluster file with pandas."""
    from fslr_b200 import cluster
    rep = cluster.choose_alignment(pd.read_csv(io.BytesIO(cluster_bed), sep="\t"))
    buf = io.StringIO()
    rep.to_csv(buf, index=False, sep="\t")
    return buf.getvalue().encode()


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_stored_fixtures(case):
    """The reference's own representative file for every stored drop-in case, from its per-read cluster / n_reads (so the
    result does not depend on the clustering's tie order)."""
    from fslr_b200 import cluster
    df = pd.DataFrame(case["rows"], columns=case["columns"])
    if case["opts"].get("filter_false"):
        df = cluster.delete_false(df)                                    # main.py:229-230
    raw = df.to_csv(index=False, sep="\t").encode()
    per_read = pd.read_csv(io.StringIO(case["expected"]["cluster_bed"]), sep="\t", dtype={"qname": str}).drop_duplicates("qname")
    pb = _parse_with_clusters(raw, dict(zip(per_read["qname"], per_read["cluster"].astype(int))),
                              dict(zip(per_read["qname"], per_read["n_reads"].astype(int))))
    try:
        assert pb.representative_bed_bytes().tobytes() == case["expected"]["representative_bed"].encode()
    finally:
        pb.close()


def _synth_bed(name, scale):
    from fslr_b200 import synth
    t = synth.make_config(name, scale)
    buf = io.StringIO()
    t.to_dataframe().to_csv(buf, index=False, sep="\t")
    return buf.getvalue().encode(), t.chr_lengths


@pytest.mark.parametrize("name,scale", [("C1", 1.0), ("C3", 0.02)])
def test_cluster_step_fast_equals_the_pandas_route(name, scale, tmp_path):
    from fslr_b200 import pipeline, synth
    raw, lens = _synth_bed(name, scale)
    base = str(tmp_path / "o")
    res = pipeline.cluster_step_fast(raw, lens, base, cluster_mask=synth.CONFIG_MASK[name])
    assert res is not None
    cl = open(base + ".mappings.cluster.bed", "rb").read()
    assert open(base + ".mappings.representative.bed", "rb").read() == _pandas_route(cl)


def test_bam_to_clusters_equals_the_pandas_route(tmp_path):
    from fslr_b200 import pipeline, synth_bam as sb
    # short references, so that alignments overlap and reads cluster; no mask (the subtelomere mask would cover them whole)
    refs, recs, primers = sb.make_alignments(1500, seed=41, refs=[("chr1", 6000), ("chr2", 5000)], p_single=0.1)
    bam = str(tmp_path / "t.bam")
    sb.write_bam(bam, refs, [sb.encode_record(*r) for r in recs])
    base = str(tmp_path / "s")
    assert pipeline.bam_to_clusters(bam, primers, base, fslr_version="9.9", cluster_mask="") is not None
    cl = open(base + ".mappings.cluster.bed", "rb").read()
    assert open(base + ".mappings.representative.bed", "rb").read() == _pandas_route(cl)


def test_integer_columns_when_every_read_is_clustered(tmp_path):
    from fslr_b200 import pipeline
    case = next(c for c in CASES if c["name"] == "all_clustered_int_columns")
    bed = tmp_path / "in.mappings.bed"
    pd.DataFrame(case["rows"], columns=case["columns"]).to_csv(bed, index=False, sep="\t")
    base = str(tmp_path / "o")
    assert pipeline.cluster_step_fast(str(bed), dict(case["chr_lengths"]), base) is not None
    assert open(base + ".mappings.representative.bed").read() == case["expected"]["representative_bed"]


def _crafted():
    """Cluster 0: A (scores 10, 20) ties B (15, 15, 15) at 15, and A's first row comes first; B's rows are interleaved with
    A's.  Cluster 1: negative scores, C (-5, -6) beats D (-7).  Cluster 2: E has 20 000 rows summing to 1, a mean of 5e-05
    that needs scientific notation, and beats F (-1).  Cluster 3: G alone, so the columns are floats."""
    rows = [("A", 10), ("B", 15), ("B", 15), ("A", 20), ("B", 15), ("D", -7), ("C", -5), ("C", -6), ("F", -1)]
    rows += [("E", 1 if i == 0 else 0) for i in range(20000)] + [("G", 3)]
    lines = [HEADER] + ["chr1\t%d\t%d\t%s\t2\t100\t0\t100\t%d" % (1000 + i, 1100 + i, q, s) for i, (q, s) in enumerate(rows)]
    raw = ("\n".join(lines) + "\n").encode()
    cluster = {"A": 0, "B": 0, "C": 1, "D": 1, "E": 2, "F": 2, "G": 3}
    n_reads = {"A": 2, "B": 2, "C": 2, "D": 2, "E": 2, "F": 2, "G": 1}
    return raw, cluster, n_reads


def test_ties_negative_scores_scattered_rows_and_tiny_means():
    raw, cluster, n_reads = _crafted()
    pb = _parse_with_clusters(raw, cluster, n_reads)
    try:
        got = pb.representative_bed_bytes().tobytes()
        assert got == _pandas_route(pb.cluster_bed_bytes().tobytes())
    finally:
        pb.close()
    lines = got.decode().splitlines()
    assert lines[0] == HEADER + "\tcluster\tn_reads\tavg_alignment_score"
    body = [ln.split("\t") for ln in lines[1:]]
    assert [(f[3], f[-3], f[-2], f[-1]) for f in body if f[3] != "E"] == [
        ("A", "0.0", "2.0", "15.0"), ("A", "0.0", "2.0", "15.0"), ("C", "1.0", "2.0", "-5.5"), ("C", "1.0", "2.0", "-5.5"),
        ("G", "3.0", "1.0", "3.0")]
    e = [f for f in body if f[3] == "E"]
    assert len(e) == 20000 and all(f[-1] == "5e-05" for f in e)


def test_size_query_matches_the_rendering():
    from fslr_b200 import _native
    raw, cluster, n_reads = _crafted()
    pb = _parse_with_clusters(raw, cluster, n_reads)
    try:
        n = C.c_int64(-1)
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        pb.engine._check(pb.engine.lib.fslrc_tsv_write_representative_bed(pb.engine.ctx, pb.out_cluster.data_ptr(),
                                                                          pb.out_n_reads.data_ptr(), None, 0, C.byref(n), stream))
        assert n.value == pb.representative_bed_bytes().nbytes
        small = np.zeros(n.value - 1, np.uint8)
        with pytest.raises(_native.FslrError):
            pb.engine._check(pb.engine.lib.fslrc_tsv_write_representative_bed(
                pb.engine.ctx, pb.out_cluster.data_ptr(), pb.out_n_reads.data_ptr(), small.ctypes.data, small.shape[0], C.byref(n), stream))
    finally:
        pb.close()


def test_errors():
    from fslr_b200 import _native, tsv
    raw, cluster, n_reads = _crafted()
    no_score = b"\n".join(ln.rsplit(b"\t", 1)[0] for ln in raw.split(b"\n")[:-1]) + b"\n"
    pb = tsv.read_mappings_bed(no_score, {})
    with pytest.raises(_native.FslrError) as e:                         # the reference raises KeyError
        pb.representative_bed_bytes()
    assert e.value.code == -2
    pb.close()
    for bad in (7, -1):                                                  # 7 reads: ids must lie in [0, 7)
        pb = _parse_with_clusters(raw, dict(cluster, C=bad), n_reads)
        with pytest.raises(_native.FslrError) as e:
            pb.representative_bed_bytes()
        assert e.value.code == -7
        pb.out_cluster[:pb.n_reads].clamp_(0, pb.n_reads - 1)           # the context is still usable afterwards
        assert pb.representative_bed_bytes().nbytes > 0
        pb.close()
    pb1 = _parse_with_clusters(raw, cluster, n_reads)
    pb2 = _parse_with_clusters(raw, cluster, n_reads)
    with pytest.raises(RuntimeError, match="stale"):
        pb1.representative_bed_bytes()
    pb2.close()
    with pytest.raises(RuntimeError, match="closed"):
        pb2.representative_bed_bytes()
