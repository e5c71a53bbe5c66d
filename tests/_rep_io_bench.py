"""Development measurement (not a test): `<base>.mappings.representative.bed` rendered on the GPU from the parsed table vs
the pandas route it replaced (read_csv of cluster.bed, cluster.choose_alignment, to_csv), C3-sized table (1M reads).
The two files are checked byte for byte before either is timed; parse, clustering and the cluster file are timed along
the way.  Usage: python tests/_rep_io_bench.py [scale] [repetitions]"""
import io
import subprocess
import sys
import time

import pandas as pd
import torch

sys.path.insert(0, ".")
from fslr_b200 import cluster, synth, tsv                               # noqa: E402

scale = float(sys.argv[1]) if len(sys.argv) > 1 else 1.0
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip())
t = synth.make_config("C3", scale)
buf = io.StringIO()
t0 = time.perf_counter(); t.to_dataframe().to_csv(buf, index=False, sep="\t"); raw = buf.getvalue().encode()
print("table: %d rows, %.1f MB of TSV (pandas to_csv %.1f s)" % (t.n_rows, len(raw) / 1e6, time.perf_counter() - t0))
t0 = time.perf_counter(); df = pd.read_csv(io.BytesIO(raw), sep="\t"); t_pd = time.perf_counter() - t0
print("pandas read_csv: %.2f s (%.0f MB/s)" % (t_pd, len(raw) / 1e6 / t_pd))


def pandas_route(cluster_bed):
    """cluster_step_fast's representative file before it was rendered on the device."""
    t0 = time.perf_counter(); df = pd.read_csv(io.BytesIO(cluster_bed), sep="\t")
    t1 = time.perf_counter(); rep = cluster.choose_alignment(df)
    t2 = time.perf_counter(); buf = io.StringIO(); rep.to_csv(buf, index=False, sep="\t"); out = buf.getvalue().encode()
    t3 = time.perf_counter()
    return out, (t1 - t0, t2 - t1, t3 - t2)


ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
dev_ms, wall_ms = [], []
for rep in range(reps):
    t0 = time.perf_counter()
    pb = tsv.read_mappings_bed(raw, t.chr_lengths)
    t1 = time.perf_counter()
    res = pb.cluster(cluster_mask=synth.CONFIG_MASK["C3"])
    t2 = time.perf_counter()
    out = pb.cluster_bed_bytes()
    t3 = time.perf_counter()
    print("gpu: parse %.1f ms wall (%.2f ms on the device after the upload, %.1f GB/s), cluster %.1f ms, render+download %.1f ms, %.1f MB out"
          % (1e3 * (t1 - t0), pb.parse_ms, len(raw) / 1e6 / max(pb.parse_ms, 1e-9), 1e3 * (t2 - t1), 1e3 * (t3 - t2), out.nbytes / 1e6))
    cl = out.tobytes()                                                  # (the representative file reuses the staging buffer)
    torch.cuda.synchronize()
    t4 = time.perf_counter(); ev0.record()
    rb = pb.representative_bed_bytes()
    ev1.record(); ev1.synchronize(); t5 = time.perf_counter()
    dev_ms.append(ev0.elapsed_time(ev1)); wall_ms.append(1e3 * (t5 - t4))
    print("gpu: representative render+download %.1f ms wall, %.1f ms between device events, %.1f MB out"
          % (wall_ms[-1], dev_ms[-1], rb.nbytes / 1e6))
    if rep == 0:
        want, _ = pandas_route(cl)
        assert rb.tobytes() == want, "device and pandas representative files differ"
        print("representative file: device bytes == pandas route bytes (%d bytes)" % len(want))
    pb.close()
pd_s = []
for rep in range(reps):
    _, parts = pandas_route(cl)
    pd_s.append(sum(parts))
    print("pandas route: read_csv %.2f s, choose_alignment %.2f s, to_csv %.2f s, total %.2f s" % (*parts, pd_s[-1]))
print("representative file, %d repetitions: device %.1f-%.1f ms wall (%.1f-%.1f ms device events), pandas %.2f-%.2f s"
      % (reps, min(wall_ms), max(wall_ms), min(dev_ms), max(dev_ms), min(pd_s), max(pd_s)))
