"""Drop-in for the functions /root/reference/fslr/main.py:227-244 calls in /root/reference/fslr/cluster.py.

Same names, positional signatures and error behaviour (ZeroDivisionError for zero divisors), so the clustering block
of main.py runs unchanged with `from fslr_b200 import cluster`:

    bed_file, chr_lengths, chromosome_mask, chrom_to_num_map = cluster.rename_chromosomes(bed_file, chr_lengths, chromosome_mask)
    fillings = cluster.keep_fillings(bed_file)
    data = cluster.prepare_data(fillings, chromosome_mask, chr_lengths, threshold=500_000)
    interval_tree = cluster.build_interval_trees(data)
    match_data, network = cluster.query_interval_trees(interval_tree, data, overlap, jaccard_cutoffs, edge_threshold, qlen_diff, n_alignments_diff)
    subgraphs = cluster.get_subgraphs(network)

The intermediate objects are opaque handles (the reference only ever passes them on): all arithmetic runs in one
fused GPU call when `query_interval_trees` is reached.  `cluster_table` is the fused entry (SURVEY.md §8b).
There is no CPU path: without the CUDA library or a device these functions raise.
"""
import os

import numpy as np
import pandas as pd

from ._native import FslrError
from .engine import ClusterResult, get_engine
from .table import ClusterParams, ColumnarTable, SUBTEL_DEFAULT

TIE_ORDER = "reference"      # "reference": same permutation numpy's unstable sort yields on this host (cluster.py:114)
                             # "stable":    GPU stable radix sort (ties keep bed order)


# ---------------------------------------------------------------- host-only helpers with reference semantics
def rename_chromosomes(bed_file, chromosome_lengths, chromosome_mask):
    """cluster.py:34-43 — chrN numerically first, then the others; ids are 1-based."""
    def key(x):
        return int(x[3:]) if x[:3] == "chr" and x[3:].isdigit() else float("inf")
    names = sorted(set(bed_file["chrom"].unique().tolist()), key=key)
    to_num = {name: i + 1 for i, name in enumerate(names)}
    chr_lengths = {to_num.get(k): v for k, v in chromosome_lengths.items()}
    bed_file["chrom"] = bed_file["chrom"].map(to_num)
    chromosome_mask = [to_num.get(x) if x != "subtelomere" else x for x in chromosome_mask]
    return bed_file, chr_lengths, chromosome_mask, to_num


def chrom_to_str(bed_df, chromosome_to_numeric_map):
    """cluster.py:46-49"""
    inv = {v: k for k, v in chromosome_to_numeric_map.items()}
    bed_df["chrom"] = bed_df["chrom"].map(inv)
    return bed_df


def delete_false(bed_file):
    """cluster.py:80-86 (--filter-false)"""
    return bed_file[~bed_file["qname"].str.contains("False")]


def get_chromosome_lengths(bam_path):
    """cluster.py:173-175 without pysam (SURVEY §8f row 3): {reference name: length} from the BAM header.  The file is
    mapped, not read, and the BGZF reader of mapping_info inflates only the blocks the header spans, each checked against
    its CRC32 and ISIZE as htslib checks it (ValueError on a mismatch, naming the block)."""
    import mmap
    from .mapping_info import bgzf_header_prefix
    with open(bam_path, "rb") as f:
        if os.fstat(f.fileno()).st_size == 0:
            raise ValueError("%s: empty file, not a BAM file" % bam_path)
        raw = mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ)           # (closed when the last view of it goes)
    try:
        refs, _ = bgzf_header_prefix(raw)
    except ValueError as e:
        raise ValueError("%s: %s" % (bam_path, e)) from None
    return dict(refs)


def reference_order_of_starts(start):
    """The permutation `sort_values('start')` (cluster.py:114) applies to a fillings frame whose `start` column is `start`
    (in bed order).  pandas hands an int64 column to numpy's default quicksort, which is unstable and whose tie order
    depends on the CPU numpy dispatches to; calling the same routine on the same int64 column reproduces the reference's
    tie order on this host exactly.  The one definition of "reference tie order" for every route."""
    start = np.asarray(start).astype(np.int64)              # the dtype read_csv gives the reference: ties are sorted as int64
    return pd.DataFrame({"start": start}).sort_values("start").index.to_numpy().astype(np.int32)


def reference_tie_order(table: ColumnarTable):
    """reference_order_of_starts of the fillings frame keep_fillings (cluster.py:14-31) makes of a host table."""
    rid = table.read_id
    A = rid.shape[0]
    idx = np.arange(A)
    first = np.full(table.n_reads, A, dtype=np.int64)
    last = np.full(table.n_reads, -1, dtype=np.int64)
    np.minimum.at(first, rid, idx)
    np.maximum.at(last, rid, idx)
    keep = (idx != first[rid]) & (idx != last[rid])
    return reference_order_of_starts(np.minimum(table.rstart[keep], table.rend[keep]))


# ---------------------------------------------------------------- opaque handles
class Fillings:
    """Returned by keep_fillings (cluster.py:14-31): the table whose first/last row per read will be dropped on the GPU."""

    def __init__(self, bed_file):
        self.bed_file = bed_file

    def __len__(self):
        return len(self.bed_file)


class PreparedData:
    """Returned by prepare_data (cluster.py:109-121)."""

    def __init__(self, fillings, cluster_mask, chromosome_lengths, threshold):
        self.bed_file = fillings.bed_file
        self.cluster_mask = list(cluster_mask) if cluster_mask else []
        self.chromosome_lengths = dict(chromosome_lengths)
        self.threshold = threshold


class IntervalIndex:
    """Returned by build_interval_trees (cluster.py:124-130); the sorted per-chromosome index lives on the GPU."""

    def __init__(self, data):
        self.data = data


class ClusterGraph:
    """Stands in for the nx.Graph of cluster.py:192,221: main.py only calls number_of_nodes() on it."""

    def __init__(self, table, result: ClusterResult):
        self.table, self.result = table, result

    def number_of_nodes(self):
        return int(self.result.stats["clustered_reads"])

    def number_of_edges(self):
        return int(self.result.stats["edges"])

    def edges(self):
        """The graph's edges as (query1, query2) qname pairs, in match_df's row order.  Needs the graph to have been
        captured: query_interval_trees(..., with_matches=True)."""
        e = self.result.edges
        if e is None:
            raise RuntimeError("the similarity graph was not captured: call query_interval_trees(..., with_matches=True)")
        q = self.table.qnames
        return [(q[a], q[b]) for a, b in zip(e.read1.tolist(), e.read2.tolist())]


def keep_fillings(bed_file):
    return Fillings(bed_file)


def prepare_data(bed_df, cluster_mask, chromosome_lengths, threshold=SUBTEL_DEFAULT):
    if not isinstance(bed_df, Fillings):
        raise TypeError("prepare_data expects the object keep_fillings returned")
    return PreparedData(bed_df, cluster_mask, chromosome_lengths, threshold)


def build_interval_trees(data):
    return IntervalIndex(data)


def _run(table, params, tie_order, device, edges=False):
    order = reference_tie_order(table) if tie_order == "reference" else None
    try:
        return get_engine(device).cluster(table, params, order=order, edges=edges)
    except FslrError as e:
        if e.code == -3:
            raise ZeroDivisionError(str(e))      # what cluster.py:135,179,181 raise
        raise


def match_frame(qnames, edges):
    """cluster.py:226's match_df from an EdgeList: query1, query2 (qnames), jaccard_similarity (float64)."""
    if edges is None:
        return pd.DataFrame(columns=["query1", "query2", "jaccard_similarity"])
    q = np.asarray(qnames, dtype=object)
    return pd.DataFrame({"query1": q[edges.read1], "query2": q[edges.read2], "jaccard_similarity": edges.jaccard})


def query_interval_trees(interval_trees, data, overlap_cutoff, jaccard_threshold, edge_threshold, qlen_diff, diff,
                         tie_order=None, device=0, with_matches=False):
    """cluster.py:187-227.  Returns (match_df, G).  main.py:242 ignores match_df, so by default it comes back empty;
    with_matches=True fills it with one row per edge of the similarity graph (query1 = the read whose query tested the
    pair, query2, jaccard_similarity), sorted by the order in which cluster.py:197 visits query1 and query2, and lets
    G.edges() list the same pairs."""
    d = data if isinstance(data, PreparedData) else interval_trees.data
    table = ColumnarTable.from_dataframe(d.bed_file, {k: v for k, v in d.chromosome_lengths.items() if k is not None})
    masked = np.zeros(table.n_chrom, dtype=np.uint8)
    sub = False
    for item in d.cluster_mask:                                   # cluster.py:96,98
        if item == "subtelomere":
            sub = True
        elif item in table.chrom_names:
            masked[table.chrom_names.index(item)] = 1
    params = ClusterParams(jaccard_cutoffs=[float(x) for x in jaccard_threshold], overlap=float(overlap_cutoff),
                           n_alignment_diff=float(diff), qlen_diff=float(qlen_diff), chrom_masked=masked,
                           mask_subtelomere=sub, subtel=int(d.threshold), edge_threshold=int(edge_threshold))
    res = _run(table, params, tie_order or TIE_ORDER, device, edges=with_matches)
    return match_frame(table.qnames, res.edges), ClusterGraph(table, res)


def get_subgraphs(G):
    """cluster.py:230-234 — list of sets of qnames, in the order networkx would list the components."""
    res, table = G.result, G.table
    n_cl = int(res.stats["components"])
    groups = [set() for _ in range(n_cl)]
    idx = np.nonzero(res.cluster < n_cl)[0] if n_cl else []
    for r in idx:
        groups[int(res.cluster[r])].add(table.qnames[r])
    return groups


# ---------------------------------------------------------------- fused entry
def cluster_table(table, chr_lengths=None, cluster_mask="subtelomere", jaccard_cutoffs="1,1,0.66,0.66,0.66,0.5",
                  overlap=0.8, n_alignment_diff=0.25, qlen_diff=0.04, edge_threshold=10, subtel=SUBTEL_DEFAULT,
                  order=None, tie_order=None, device=0, edges=False) -> ClusterResult:
    """table: ColumnarTable or a DataFrame as read at main.py:209 (then chr_lengths is the BAM-header dict).
    Returns per-read-id `cluster` / `n_reads` (read id = order of first appearance of qname); edges=True adds the
    similarity graph (ClusterResult.edges)."""
    if not isinstance(table, ColumnarTable):
        table = ColumnarTable.from_dataframe(table, chr_lengths or {})
    params = ClusterParams.from_options(table, cluster_mask, jaccard_cutoffs, overlap, n_alignment_diff, qlen_diff,
                                        edge_threshold, subtel)
    if order is not None:
        return get_engine(device).cluster(table, params, order=order, edges=edges)
    return _run(table, params, tie_order or TIE_ORDER, device, edges=edges)


def choose_alignment(bed_file, device=0):
    """cluster.py:237-254 — the rows of the read with the highest mean alignment_score per cluster (first on ties), computed
    on the GPU (fslrc_choose_alignment_host).  Like the reference it adds the `avg_alignment_score` column to `bed_file`."""
    rid, _ = pd.factorize(bed_file["qname"], sort=False)
    score = bed_file["alignment_score"].to_numpy()
    if not np.all(np.isfinite(score)) or np.any(score != np.round(score)) or np.abs(score).max(initial=0) >= 2**31:
        raise ValueError("alignment_score must be integer valued (collect_mapping_info.py writes the AS tag)")
    n_reads = int(rid.max()) + 1 if rid.size else 0
    first_row = np.full(n_reads, rid.shape[0], dtype=np.int64)
    np.minimum.at(first_row, rid, np.arange(rid.shape[0]))
    cid, cvals = pd.factorize(bed_file["cluster"].to_numpy()[first_row], sort=False)
    is_rep, _ = get_engine(device).choose_alignment(rid, score.astype(np.int64), cid, len(cvals))
    sums = np.bincount(rid, weights=score.astype(np.float64), minlength=n_reads)
    bed_file["avg_alignment_score"] = (sums / np.maximum(np.bincount(rid, minlength=n_reads), 1))[rid]   # the column the reference adds
    return bed_file[is_rep[rid].astype(bool)]
