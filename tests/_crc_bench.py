"""Dev script (GPU box): the cost of the BGZF CRC32 check on the device BAM route, on the 200k-read BAM of
tests/_bam_bench.py (10 copies: ~5 000 blocks, 298 MB inflated).  python tests/_crc_bench.py [copies] [reps] [--parse-only]
-> one JSON line.  With --parse-only and FSLR_B200_LIB naming a build of the library without the check, the same
timings compare the two.

- k_bgzf_crc and k_inflate device times from torch.profiler (CUDA activities) in a run of their own;
- inflated bytes / k_bgzf_crc time, against the 7.7 TB/s HBM3e bandwidth of a B200's data sheet;
- wall time and parse_ms (device events around the open's kernels) of read_bam_table(path) after a warm-up;
- whether mappings.bed equals the host-inflate route's bytes."""
import json
import os
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch                                                            # noqa: E402
from torch.profiler import ProfilerActivity, profile                    # noqa: E402

from fslr_b200 import mapping_info as mi                                # noqa: E402
from tests import bgzf_cases as bc                                      # noqa: E402

args = [a for a in sys.argv[1:] if not a.startswith("--")]
copies = int(args[0]) if args else 10
reps = int(args[1]) if len(args) > 1 else 7
parse_only = "--parse-only" in sys.argv           # only the wall / parse_ms timings: runs on a library without the check too
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                      text=True).stdout.strip().splitlines()
raw, primers = bc.bench_bam(copies)
path = os.path.join(tempfile.mkdtemp(), "big.bam")
open(path, "wb").write(raw)
n_blocks = len(bc.block_offsets(raw))

a = mi.read_bam_table(path, None, primers, device_inflate=False)       # reference bytes: host zlib inflate
want = a.mappings_bed_bytes("9.9").tobytes()
inflated = int(a._stream().shape[0])
a.close()

t = mi.read_bam_table(path, None, primers)                              # warm-up, and the output check
same = t.mappings_bed_bytes("9.9").tobytes() == want
fallback = int(t.info.reserved)
t.close()

wall, parse = [], []
for _ in range(reps):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    t = mi.read_bam_table(path, None, primers)                          # (returns after a stream synchronise)
    wall.append((time.perf_counter() - t0) * 1e3)
    parse.append(t.parse_ms)
    t.close()
if parse_only:
    print(json.dumps({"card": card, "lib": os.path.basename(os.environ.get("FSLR_B200_LIB", "libfslr_b200.so")), "read_bam_table_wall_ms": [round(x, 3) for x in wall],
                      "parse_ms": [round(x, 3) for x in parse], "same_bytes_as_host_inflate": bool(same)}))
    sys.exit(0)

with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(3):
        mi.read_bam_table(path, None, primers).close()
    torch.cuda.synchronize()
kern = {}
for ev in prof.key_averages():
    for name in ("k_bgzf_crc", "k_inflate"):
        if name in ev.key:
            kern[name] = {"calls": ev.count, "ms_per_call": ev.device_time_total / ev.count / 1e3}
crc_ms = kern["k_bgzf_crc"]["ms_per_call"]
out = {"card": card, "reads": 20000 * copies, "bam_MB": len(raw) / 1e6, "inflated_MB": inflated / 1e6, "bgzf_blocks": n_blocks,
       "kernels": kern, "crc_GB_per_s": inflated / (crc_ms * 1e-3) / 1e9,
       "crc_share_of_7.7TB_per_s": inflated / (crc_ms * 1e-3) / 7.7e12,
       "crc_share_of_inflate": crc_ms / kern["k_inflate"]["ms_per_call"],
       "read_bam_table_wall_ms": [round(x, 3) for x in wall], "parse_ms": [round(x, 3) for x in parse],
       "host_walk_fallback": fallback, "same_bytes_as_host_inflate": bool(same)}
print(json.dumps(out))
