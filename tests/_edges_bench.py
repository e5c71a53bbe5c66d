"""Development measurement (not a test): the cost of the edge export (fslrc_set_edge_capture).
1. C4 (10M reads), resident step: capture off against capture on, alternated; the capture-on time includes the export
   kernels, the sort and fslrc_edges into device buffers (not the download to the host).  Host clock around a synchronised
   call.
2. C3 (1M reads), file to files through pipeline.cluster_step_fast, without and with `edges`; the edges file is checked
   against the CPU oracle's rows first.
Usage: python tests/_edges_bench.py [repetitions]"""
import ctypes as C
import io
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np
import pandas as pd
import torch

sys.path.insert(0, ".")
from fslr_b200 import _native, pipeline, synth                          # noqa: E402
from fslr_b200.engine import DeviceTable, get_engine                    # noqa: E402
from fslr_b200.table import ClusterParams, ColumnarTable                # noqa: E402
from tests.oracle_edges import oracle_cluster_edges                     # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip())
eng = get_engine(0)

# ---- 1. C4 resident step
t = ColumnarTable.from_synth(synth.make_config("C4"))
p = ClusterParams.from_options(t, cluster_mask=synth.CONFIG_MASK["C4"])
d = DeviceTable(t, eng.device)
pp, tt = eng._params(t, p), eng._table(d)
stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
bufs = None


def step(capture):
    global bufs
    eng._set_capture(capture)
    st = _native.Stats()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    eng._check(eng.lib.fslrc_cluster_device(eng.ctx, C.byref(tt), C.byref(pp), d.out_cluster.data_ptr(), d.out_n_reads.data_ptr(),
                                            C.byref(st), stream))
    n = C.c_int64()
    if capture:
        eng._check(eng.lib.fslrc_edges(eng.ctx, None, None, None, 0, C.byref(n), stream))
        if bufs is None or bufs[0].numel() < n.value:
            bufs = [torch.empty(n.value, dtype=dt, device=eng.device) for dt in (torch.int32, torch.int32, torch.float64)]
        eng._check(eng.lib.fslrc_edges(eng.ctx, bufs[0].data_ptr(), bufs[1].data_ptr(), bufs[2].data_ptr(), n.value, C.byref(n), stream))
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0), st.edges, n.value


for cap in (False, True, False, True):
    step(cap)
ref = d.out_cluster[:t.n_reads].cpu().numpy().copy()
times = {False: [], True: []}
for r in range(reps):
    for cap in (False, True):
        ms, ne, n = step(cap)
        assert np.array_equal(d.out_cluster[:t.n_reads].cpu().numpy(), ref)
        assert not cap or n == ne
        times[cap].append(ms)
print("C4 resident step: %d reads, %d edges" % (t.n_reads, ne))
for cap in (False, True):
    v = sorted(times[cap])
    print("  capture %-3s: min %.2f  median %.2f  max %.2f ms  (%s)" % ("on" if cap else "off", v[0], v[len(v) // 2], v[-1],
                                                                     " ".join("%.2f" % x for x in times[cap])))
eng._set_capture(False)
del d, bufs
torch.cuda.empty_cache()

# ---- 2. C3 file to files
t = synth.make_config("C3", 1.0)
buf = io.StringIO()
t.to_dataframe().to_csv(buf, index=False, sep="\t")
raw = buf.getvalue().encode()
del buf
mask = synth.CONFIG_MASK["C3"]
tmp = tempfile.mkdtemp(prefix="fslr_edges_bench_")
try:
    bed = os.path.join(tmp, "in.mappings.bed")
    with open(bed, "wb") as f:
        f.write(raw)
    ef = os.path.join(tmp, "edges.tsv")
    pipeline.cluster_step_fast(bed, t.chr_lengths, os.path.join(tmp, "o"), cluster_mask=mask, edges=ef)
    ct = ColumnarTable.from_dataframe(pd.read_csv(io.BytesIO(raw), sep="\t"), t.chr_lengths)
    _, _, ost, (o1, o2, oj) = oracle_cluster_edges(ct, ClusterParams.from_options(ct, cluster_mask=mask))
    got = pd.read_csv(ef, sep="\t", dtype={"query1": str, "query2": str}, float_precision="round_trip")
    q = np.asarray(ct.qnames, dtype=object)
    assert set(zip(got.query1, got.query2, got.jaccard_similarity.to_numpy().view(np.uint64).tolist())) == \
        set(zip(q[o1], q[o2], oj.view(np.uint64).tolist())) and len(got) == ost["edges"]
    print("C3 file to files: %d rows, %d reads, %.1f MB TSV; edges file: %d edges, %.1f MB, equal to the oracle's rows"
          % (t.n_rows, t.n_reads, len(raw) / 1e6, len(got), os.path.getsize(ef) / 1e6))
    times = {False: [], True: []}
    for r in range(reps + 1):
        for with_edges in (False, True):
            t0 = time.perf_counter()
            pipeline.cluster_step_fast(bed, t.chr_lengths, os.path.join(tmp, "o"), cluster_mask=mask, edges=ef if with_edges else None)
            if r:
                times[with_edges].append(time.perf_counter() - t0)
    for k in (False, True):
        v = sorted(times[k])
        print("  cluster_step_fast %-13s: min %.3f  median %.3f  max %.3f s" % ("with --edges" if k else "without", v[0], v[len(v) // 2], v[-1]))
finally:
    shutil.rmtree(tmp)
