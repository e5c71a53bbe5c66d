"""Development measurement (not a test): the cost of tie_order="reference" on the GPU file path.  C3-sized table (1M reads):
the parse (read_mappings_bed), fslrc_filling_starts (device events), the download of the start column + the host sort
(cluster.reference_order_of_starts, the reference's pandas call) + the upload of the order (wall), the clustering with that
order (general ingest) against the stable one (fast ingest), and both renderings.  Both device files are checked byte for
byte against the pandas route (pipeline.cluster_step, tie_order="reference") before anything is timed.
Repetition 0 includes the first launches of every kernel.  The render times run from the event before the call to one
recorded after the bytes were copied out of the staging buffer, so they include the download and that host copy.
Usage: python tests/_tie_order_bench.py [scale] [repetitions]"""
import io
import os
import shutil
import subprocess
import sys
import tempfile
import time

import torch

sys.path.insert(0, ".")
from fslr_b200 import pipeline, synth, tsv                              # noqa: E402
from fslr_b200.cluster import reference_order_of_starts                 # noqa: E402

scale = float(sys.argv[1]) if len(sys.argv) > 1 else 1.0
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip())
t = synth.make_config("C3", scale)
buf = io.StringIO()
t.to_dataframe().to_csv(buf, index=False, sep="\t")
raw = buf.getvalue().encode()
del buf
mask = synth.CONFIG_MASK["C3"]
print("table: %d rows, %d reads, %.1f MB of TSV" % (t.n_rows, t.n_reads, len(raw) / 1e6))
tmp = tempfile.mkdtemp(prefix="fslr_tie_bench_")
try:
    bed = os.path.join(tmp, "in.mappings.bed")
    with open(bed, "wb") as f:
        f.write(raw)
    t0 = time.perf_counter()
    pipeline.cluster_step(bed, t.chr_lengths, cluster_mask=mask, tie_order="reference", out_base=os.path.join(tmp, "ref"))
    print("pandas route, reference tie order (for the byte check): %.1f s" % (time.perf_counter() - t0))
    want = [open(os.path.join(tmp, "ref" + f), "rb").read() for f in (".mappings.cluster.bed", ".mappings.representative.bed")]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(8)]
    rows = []
    for rep in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pb = tsv.read_mappings_bed(raw, t.chr_lengths)
        t1 = time.perf_counter()
        eng = pb.engine
        ev[0].record()
        start = eng.filling_starts(pb)
        ev[1].record(); ev[1].synchronize()
        t2 = time.perf_counter()
        h = start.cpu().numpy()
        t3 = time.perf_counter()
        order_h = reference_order_of_starts(h)
        t4 = time.perf_counter()
        order = torch.from_numpy(order_h).to(eng.device)
        torch.cuda.synchronize()
        t5 = time.perf_counter()
        pb._reference_order = order                                     # (what cluster(tie_order="reference") computes and keeps)
        ev[2].record()
        pb.cluster(cluster_mask=mask, tie_order="stable")
        ev[3].record()
        pb.cluster(cluster_mask=mask, tie_order="reference")
        ev[4].record()
        cl = pb.cluster_bed_bytes().tobytes()
        ev[5].record()
        rb = pb.representative_bed_bytes().tobytes()
        ev[6].record(); ev[6].synchronize()
        t6 = time.perf_counter()
        assert cl == want[0] and rb == want[1], "device and pandas files differ"
        r = dict(wall_read=1e3 * (t1 - t0), parse=pb.parse_ms, starts=ev[0].elapsed_time(ev[1]), wall_starts=1e3 * (t2 - t1),
                 down=1e3 * (t3 - t2), sort=1e3 * (t4 - t3), up=1e3 * (t5 - t4), host=1e3 * (t5 - t2),
                 stable=ev[2].elapsed_time(ev[3]), ref=ev[3].elapsed_time(ev[4]), r_cl=ev[4].elapsed_time(ev[5]),
                 r_rep=ev[5].elapsed_time(ev[6]), n_fill=len(h), wall_total=1e3 * (t6 - t0))
        rows.append(r)
        print("rep %d: read_mappings_bed %.1f ms wall (parse %.2f ms events) | fslrc_filling_starts %.3f ms events (%d fillings) | "
              "download %.1f + host sort %.1f + upload %.1f = %.1f ms wall | cluster stable %.2f ms, reference %.2f ms events | "
              "cluster.bed %.2f ms, representative.bed %.2f ms events (render, download, copy to bytes) | files == pandas route (reference)"
              % (rep, r["wall_read"], r["parse"], r["starts"], r["n_fill"], r["down"], r["sort"], r["up"], r["host"], r["stable"],
                 r["ref"], r["r_cl"], r["r_rep"]))
        pb.close()
    # the whole route as a user runs it, both modes (parse, clustering, both files written)
    for mode in ("stable", "reference"):
        ts = []
        for rep in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            pipeline.cluster_step_fast(bed, t.chr_lengths, os.path.join(tmp, mode), cluster_mask=mask, tie_order=mode)
            ts.append(time.perf_counter() - t0)
        print("cluster_step_fast(tie_order=%r), file to files: %s s" % (mode, ", ".join("%.3f" % x for x in ts)))
    assert [open(os.path.join(tmp, "reference" + f), "rb").read() for f in (".mappings.cluster.bed", ".mappings.representative.bed")] == want
    rng_ = lambda k: (min(r[k] for r in rows[1:] or rows), max(r[k] for r in rows[1:] or rows))
    print("repetitions 1-%d (min-max): parse %.2f-%.2f ms, fslrc_filling_starts %.3f-%.3f ms (events); download %.1f-%.1f, host sort "
          "%.1f-%.1f, upload %.1f-%.1f ms (wall); cluster stable %.2f-%.2f ms, reference %.2f-%.2f ms; cluster.bed %.2f-%.2f ms, "
          "representative.bed %.2f-%.2f ms (events)"
          % (reps - 1, *rng_("parse"), *rng_("starts"), *rng_("down"), *rng_("sort"), *rng_("up"), *rng_("stable"), *rng_("ref"),
             *rng_("r_cl"), *rng_("r_rep")))
finally:
    shutil.rmtree(tmp, ignore_errors=True)
