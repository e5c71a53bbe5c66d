"""The clustering block of /root/reference/fslr/main.py:190-352 around the B200 library: reads `<base>.mappings.bed`,
clusters on the GPU, writes `<base>.mappings.cluster.bed` and `<base>.mappings.representative.bed` with the same
columns and dtypes (float `cluster` / `n_reads`, main.py:334-349).  `chr_lengths` replaces the BAM-header lookup of
main.py:225 (cluster.get_chromosome_lengths needs pysam).
"""
import json
import sys

import numpy as np
import pandas as pd

from . import cluster as gcluster
from .table import ColumnarTable


def cluster_step_fast(bed_path, chr_lengths, out_base, cluster_mask="subtelomere", jaccard_cutoffs="1,1,0.66,0.66,0.66,0.5",
                      overlap=0.8, n_alignment_diff=0.25, qlen_diff=0.04, representative=True, filter_false=False, device=0,
                      tie_order="stable", edges=None):
    """The same block with the table never leaving the GPU between the file bytes and the output bytes (fslr_b200.tsv):
    GPU TSV parse -> clustering on the device-resident columns -> GPU rendering of `<out_base>.mappings.cluster.bed` and
    (representative=True) `<out_base>.mappings.representative.bed`.
    filter_false drops the reads whose qname contains "False" (main.py:229-230) on the device, after the parse.
    tie_order: "stable" (default) orders equal starts with the GPU's stable sort (ids equal the reference's whenever its
    unstable sort keeps ties in table order, the partition always); "reference" uses the permutation fslr's own
    `sort_values('start')` gives on this host (a host sort of the device-built start column, see ParsedBed.cluster), so
    both files are numbered as fslr numbers them.
    edges: a path for the similarity graph (cluster.py:226's match_df, as to_csv(sep="\t", index=False) writes it), rendered
    on the device; written also on the early return, where it holds only the header.  Returns the ClusterResult, or None
    for main.py:247-249's early return."""
    from . import tsv
    print("Making clusters", file=sys.stderr)                                    # main.py:207
    pb = tsv.read_mappings_bed(bed_path, chr_lengths, device=device, filter_false=filter_false)   # main.py:209, 229-230
    try:
        res = pb.cluster(cluster_mask=cluster_mask, jaccard_cutoffs=jaccard_cutoffs, overlap=overlap,
                         n_alignment_diff=n_alignment_diff, qlen_diff=qlen_diff, tie_order=tie_order, edges=bool(edges))
        if edges:
            pb.write_edges(edges)
        if res.no_clusters:
            print("No clusters were found.", file=sys.stderr)                    # main.py:247-249
            return None
        pb.write_cluster_bed(f"{out_base}.mappings.cluster.bed")                 # main.py:349
        if representative:                                                       # main.py:351-352
            pb.write_representative_bed(f"{out_base}.mappings.representative.bed")
        return res
    finally:
        pb.close()


def bam_to_clusters(bam_path, primers, out_base, regions_path=None, fslr_version=None, device=0, **cluster_options):
    """main.py:181-183 + main.py:190-352 without the table ever being parsed on the host: `<base>.bwa_dodi.bam` ->
    `<out_base>.mappings.bed` (fslr_b200.mapping_info, the GPU stand-in for collect_mapping_info.mapping_info) ->
    `<out_base>.mappings.cluster.bed` (+ representative).  The chromosome lengths come from the same BAM header
    (cluster.py:173-175).  primers: {name: sequence} as main.py:69 builds it from primers.csv.  cluster_options go to
    cluster_step_fast (tie_order included); with filter_false=True the written mappings.bed still holds every read, as in
    main.py."""
    from . import mapping_info as mi
    t = mi.read_bam_table(bam_path, regions_path, primers, device=device)
    try:
        bed = t.mappings_bed_bytes(fslr_version)
        lengths = {n: int(l) for n, l in zip(t.chrom_names, t.chrom_len) if l > 0}
    finally:
        t.close()
    bed.tofile(f"{out_base}.mappings.bed")                                       # collect_mapping_info.py:181
    return cluster_step_fast(bed.tobytes(), lengths, out_base, device=device, **cluster_options)


def cluster_step(bed_file, chr_lengths, cluster_mask="subtelomere", jaccard_cutoffs="1,1,0.66,0.66,0.66,0.5", overlap=0.8,
                 n_alignment_diff=0.25, qlen_diff=0.04, filter_false=False, out_base=None, tie_order=None, device=0, edges=None):
    """Returns the annotated DataFrame, or None when main.py:247-249 would print "No clusters were found." and return.
    edges: a path for the similarity graph, written with match_df.to_csv(sep="\t", index=False) (header only on the
    early return)."""
    if isinstance(bed_file, str):
        bed_file = pd.read_csv(bed_file, sep="\t")                               # main.py:209
    print("Making clusters", file=sys.stderr)                                    # main.py:207
    if filter_false:
        bed_file = gcluster.delete_false(bed_file)                               # main.py:229-230
    table = ColumnarTable.from_dataframe(bed_file, chr_lengths)
    res = gcluster.cluster_table(table, cluster_mask=cluster_mask, jaccard_cutoffs=jaccard_cutoffs, overlap=overlap,
                                 n_alignment_diff=n_alignment_diff, qlen_diff=qlen_diff, tie_order=tie_order, device=device,
                                 edges=bool(edges))
    if edges:
        gcluster.match_frame(table.qnames, res.edges).to_csv(edges, sep="\t", index=False)
    if res.no_clusters:
        print("No clusters were found.", file=sys.stderr)                        # main.py:247-249
        return None
    bed_file = bed_file.copy()
    # main.py:334-342: the left merge leaves NaN on singleton rows, so the columns are floats — unless every read ended in
    # a cluster, in which case pandas keeps the integer dtype
    dt = np.float64 if bool((res.n_reads == 1).any()) else np.int64
    bed_file["cluster"] = res.cluster[table.read_id].astype(dt)
    bed_file["n_reads"] = res.n_reads[table.read_id].astype(dt)
    if out_base:
        bed_file.to_csv(f"{out_base}.mappings.cluster.bed", index=False, sep="\t")                 # main.py:349
        rep = gcluster.choose_alignment(bed_file)                                                   # main.py:351-352
        rep.to_csv(f"{out_base}.mappings.representative.bed", index=False, sep="\t")
    return bed_file


def main(argv=None):
    import argparse
    ap = argparse.ArgumentParser(description="fslr clustering step on B200 (drop-in for `fslr --skip-alignment`'s clustering block)")
    ap.add_argument("--bed", help="<base>.mappings.bed")
    ap.add_argument("--bam", help="<base>.bwa_dodi.bam: build mappings.bed on the GPU first (needs --primers-csv and --primers)")
    ap.add_argument("--primers-csv", help="primers.csv of the fslr installation (columns primer_name, primer_seq; main.py:59)")
    ap.add_argument("--primers", help="comma-separated primer names (main.py:23)")
    ap.add_argument("--regions", help="regions BED for the overlaps_region column (collect_mapping_info.py:28-36)")
    ap.add_argument("--chr-lengths", help="JSON {chrom: length}, or the <base>.bwa_dodi.bam whose header holds them (main.py:225)")
    ap.add_argument("--out-base", required=True)
    ap.add_argument("--jaccard-cutoffs", default="1,1,0.66,0.66,0.66,0.5")
    ap.add_argument("--overlap", type=float, default=0.8)
    ap.add_argument("--n-alignment-diff", type=float, default=0.25)
    ap.add_argument("--qlen-diff", type=float, default=0.04)
    ap.add_argument("--cluster-mask", default="subtelomere")
    ap.add_argument("--filter-false", action="store_true")
    ap.add_argument("--fast-io", action="store_true", help="parse the TSV and render mappings.cluster.bed on the GPU")
    ap.add_argument("--no-representative", action="store_true")
    ap.add_argument("--edges", metavar="PATH",
                    help="also write the similarity graph: one line per edge of the clustering (query1, query2, "
                         "jaccard_similarity), as fslr's match_df")
    ap.add_argument("--tie-order", choices=("stable", "reference"),
                    help="order of fillings with equal starts, which decides the cluster numbering: 'reference' numbers the "
                         "clusters exactly as fslr does on this host (a host sort of the start column), 'stable' keeps ties "
                         "in table order.  Unset: 'stable' with --fast-io and --bam, 'reference' otherwise")
    a = ap.parse_args(argv)
    tie = {} if a.tie_order is None else {"tie_order": a.tie_order}                # unset: each route's own default
    ed = {} if a.edges is None else {"edges": a.edges}
    if a.bam:
        d = pd.read_csv(a.primers_csv)
        want = set(a.primers.split(","))
        primers = {k: v for k, v in zip(d["primer_name"], d["primer_seq"]) if k in want}       # main.py:69
        bam_to_clusters(a.bam, primers, a.out_base, a.regions, cluster_mask=a.cluster_mask, jaccard_cutoffs=a.jaccard_cutoffs,
                        overlap=a.overlap, n_alignment_diff=a.n_alignment_diff, qlen_diff=a.qlen_diff,
                        representative=not a.no_representative, filter_false=a.filter_false, **tie, **ed)
        return
    if not a.bed or not a.chr_lengths:
        ap.error("--bed and --chr-lengths are required without --bam")
    lengths = gcluster.get_chromosome_lengths(a.chr_lengths) if a.chr_lengths.endswith(".bam") else json.load(open(a.chr_lengths))
    if a.fast_io:
        cluster_step_fast(a.bed, lengths, a.out_base, a.cluster_mask, a.jaccard_cutoffs, a.overlap,
                          a.n_alignment_diff, a.qlen_diff, not a.no_representative, filter_false=a.filter_false, **tie, **ed)
        return
    cluster_step(a.bed, lengths, a.cluster_mask, a.jaccard_cutoffs, a.overlap, a.n_alignment_diff,
                 a.qlen_diff, a.filter_false, a.out_base, **tie, **ed)


if __name__ == "__main__":
    main()
