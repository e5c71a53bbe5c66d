"""Development measurement (not a test): --filter-false on the GPU file path (read_mappings_bed(filter_false=True), the
clustering, both rendered files) vs the pandas route `--fast-io --filter-false` took before the filter ran on the device
(pipeline.cluster_step: read_csv, delete_false, from_dataframe, clustering, to_csv, choose_alignment, to_csv).  C3-sized
table (1M reads) with 20 % of the reads renamed so that their names contain "False".  Both device files are checked byte
for byte against the pandas route (stable tie order) before anything is timed.
Usage: python tests/_filter_io_bench.py [scale] [repetitions]"""
import io
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, ".")
from fslr_b200 import pipeline, synth, tsv                              # noqa: E402

scale = float(sys.argv[1]) if len(sys.argv) > 1 else 1.0
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip())
t = synth.make_config("C3", scale)
df = t.to_dataframe()
names = t.qnames()[np.unique(t.read_id, return_index=True)[1]]
rng = np.random.default_rng(7)
hit = rng.random(t.n_reads) < 0.2
kind = rng.integers(0, 3, t.n_reads)
names = np.array([(("False" + q, q + "_False", q[:8] + "False" + q[8:])[k] if h else q)
                  for q, h, k in zip(names.tolist(), hit.tolist(), kind.tolist())], dtype=object)
df["qname"] = names[t.read_id]
buf = io.StringIO()
t0 = time.perf_counter(); df.to_csv(buf, index=False, sep="\t"); raw = buf.getvalue().encode()
print("table: %d rows, %d reads (%d named ...False...), %.1f MB of TSV (pandas to_csv %.1f s)"
      % (t.n_rows, t.n_reads, int(hit.sum()), len(raw) / 1e6, time.perf_counter() - t0))
del df, buf
mask = synth.CONFIG_MASK["C3"]
tmp = tempfile.mkdtemp(prefix="fslr_filter_bench_")
try:
    bed = os.path.join(tmp, "in.mappings.bed")
    with open(bed, "wb") as f:
        f.write(raw)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    rows = []
    for rep in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pb = tsv.read_mappings_bed(raw, t.chr_lengths, filter_false=True)
        t1 = time.perf_counter()
        ev[0].record()
        pb.cluster(cluster_mask=mask)
        ev[1].record()
        t2 = time.perf_counter()
        cl = pb.cluster_bed_bytes().tobytes()                           # (the staging buffer is reused by the next render)
        ev[2].record()
        rb = pb.representative_bed_bytes().tobytes()
        ev[3].record(); ev[3].synchronize()
        t3 = time.perf_counter()
        r = dict(wall_read=1e3 * (t1 - t0), parse=pb.parse_ms, filt=pb.filter_ms, clus=ev[0].elapsed_time(ev[1]),
                 wall_clus=1e3 * (t2 - t1), r_cl=ev[1].elapsed_time(ev[2]), r_rep=ev[2].elapsed_time(ev[3]), wall_r=1e3 * (t3 - t2))
        rows.append(r)
        print("gpu rep %d: %d -> %d rows, %d -> %d reads | read_mappings_bed %.1f ms wall (upload included): parse %.2f ms, "
              "filter %.3f ms between device events | cluster %.2f ms events (%.1f ms wall) | cluster.bed %.2f ms, "
              "representative.bed %.2f ms events incl. download (%.1f ms wall, %.1f + %.1f MB)"
              % (rep, t.n_rows, pb.n_rows, t.n_reads, pb.n_reads, r["wall_read"], r["parse"], r["filt"], r["clus"], r["wall_clus"],
                 r["r_cl"], r["r_rep"], r["wall_r"], len(cl) / 1e6, len(rb) / 1e6))
        pb.close()
        if rep == 0:
            t0 = time.perf_counter()
            pipeline.cluster_step(bed, t.chr_lengths, cluster_mask=mask, filter_false=True, tie_order="stable",
                                  out_base=os.path.join(tmp, "stable"))
            print("pandas route, stable tie order (for the byte check): %.1f s" % (time.perf_counter() - t0))
            for got, f in ((cl, ".mappings.cluster.bed"), (rb, ".mappings.representative.bed")):
                want = open(os.path.join(tmp, "stable" + f), "rb").read()
                assert got == want, "device and pandas %s differ" % f
                print("%s: device bytes == pandas route bytes (%d bytes)" % (f, len(want)))
    t0 = time.perf_counter()
    pipeline.cluster_step(bed, t.chr_lengths, cluster_mask=mask, filter_false=True, out_base=os.path.join(tmp, "old"))
    old_s = time.perf_counter() - t0
    print("route of --fast-io --filter-false before this change (cluster_step, default tie order), once: %.1f s" % old_s)
    rng_ = lambda k: (min(r[k] for r in rows), max(r[k] for r in rows))
    print("device, %d repetitions: parse %.2f-%.2f ms, filter %.3f-%.3f ms, cluster %.2f-%.2f ms, cluster.bed %.2f-%.2f ms, "
          "representative.bed %.2f-%.2f ms (device events); read_mappings_bed %.1f-%.1f ms wall"
          % (reps, *rng_("parse"), *rng_("filt"), *rng_("clus"), *rng_("r_cl"), *rng_("r_rep"), *rng_("wall_read")))
finally:
    shutil.rmtree(tmp, ignore_errors=True)
