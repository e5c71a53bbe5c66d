"""The CPU oracle's edge list (tests/oracle_edges.py: the unmodified oracle with the edges recorded): the edges
cluster.py:220-221 adds, as (query_key, other read, jaccard).  Its connected components are its own clusters on every stored case, and asking for the list changes
nothing else.  Also the command line's routing of --edges (no GPU: the clustering is mocked)."""
import numpy as np
import pytest
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

from tests import golden_io
from tests.oracle_edges import oracle_cluster_edges


def partition_of_edges(n_reads, read1, read2):
    """Component label per read of the graph (read1, read2); -1 for reads on no edge."""
    if len(read1) == 0:
        return np.full(n_reads, -1)
    g = coo_matrix((np.ones(len(read1)), (read1, read2)), shape=(n_reads, n_reads))
    _, lab = connected_components(g, directed=False)
    on = np.zeros(n_reads, bool)
    on[read1] = on[read2] = True
    return np.where(on, lab, -1)


def same_partition(label, cluster, n_reads_col):
    """label (edges' components, -1 = on no edge) and the clustering's (cluster, n_reads) describe the same partition."""
    single = label < 0
    if not np.array_equal(single, n_reads_col == 1):
        return False
    a, b = label[~single], cluster[~single]
    pairs = set(zip(a.tolist(), b.tolist()))
    return len(pairs) == len(set(a.tolist())) == len(set(b.tolist()))


@pytest.fixture(scope="module")
def stored():
    return {f: golden_io.load(f) for f in ("small_cases.npz", "wide_cases.npz", "config_cases.npz")}


def test_case_counts(stored):
    assert [len(stored[f]) for f in ("small_cases.npz", "wide_cases.npz", "config_cases.npz")] == [415, 120, 8]


def test_oracle_edges_give_its_clusters(stored):
    from oracle import oracle as orc
    bad = []
    for f, cases in stored.items():
        for c in cases:
            cl, nr, st = orc.oracle_cluster(c.table, c.params, order=c.order)
            cl2, nr2, st2, (r1, r2, jac) = oracle_cluster_edges(c.table, c.params, order=c.order)
            ok = (np.array_equal(cl, cl2) and np.array_equal(nr, nr2) and st == st2 and len(r1) == st["edges"]
                  and r1.dtype == np.int32 and jac.dtype == np.float64 and np.all((jac > 0) & (jac <= 1)))
            ok = ok and (st["no_clusters"] == 1) == (len(r1) == 0)
            ok = ok and same_partition(partition_of_edges(c.table.n_reads, r1, r2), cl, nr)
            if not c.no_clusters:                                     # and the reference's stored ids
                ok = ok and np.array_equal(cl, c.expected[0])
            key = set(zip(np.minimum(r1, r2).tolist(), np.maximum(r1, r2).tolist()))
            ok = ok and len(key) == len(r1) and not np.any(r1 == r2)
            if not ok:
                bad.append("%s/%s" % (f, c.name))
    assert not bad, bad[:10]


def test_oracle_edges_are_in_query_order(stored):
    """The oracle adds the edges of one query read together, query reads in turn: read1 never comes back once left."""
    c = golden_io.load("config_cases.npz")[0]
    _, _, _, (r1, _, _) = oracle_cluster_edges(c.table, c.params, order=c.order)
    runs = r1[np.r_[True, r1[1:] != r1[:-1]]]
    assert len(runs) == len(set(runs.tolist())) and len(r1) > 100


def _cli_calls(tmp_path, monkeypatch, extra):
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
    pipeline.main(bed + ["--fast-io"] + extra)
    pipeline.main(["--bam", "x.bam", "--primers-csv", str(pcsv), "--primers", "21q1", "--out-base", "o"] + extra)
    pipeline.main(bed + extra)
    assert [c[0] for c in calls] == ["fast", "bam", "pandas"]
    return calls


def test_cli_routes_edges(tmp_path, monkeypatch):
    calls = _cli_calls(tmp_path, monkeypatch, ["--edges", "g.tsv", "--tie-order", "reference"])
    assert all(c[2]["edges"] == "g.tsv" and c[2]["tie_order"] == "reference" for c in calls)
    assert all("edges" not in c[2] for c in _cli_calls(tmp_path, monkeypatch, []))
