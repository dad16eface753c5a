"""Throughput of the navigation queries on the device SdBG (not a pytest file).
usage: gpu_sdbg_query_time.py N_READS [k]   -> one JSON line

The graph of N_READS seeded metagenome reads of 150 bp (m = 2) is built on the device.  Every edge op runs on a batch of
all edges, LOOKUP and LABEL on a batch of all nodes (their labels, read back from LABEL); one warm-up pass, then PASSES
timed passes between CUDA events on the graph's stream, the median is reported.  LOOKUP is timed with and without the
lv1 bucket (MGTA_SQ_LV1=0: the f block of the last character)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import datasets  # noqa: E402
from megagta_b200 import cabi  # noqa: E402

PASSES = 3
n = int(sys.argv[1])
k = int(sys.argv[2]) if len(sys.argv) > 2 else 31
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
out = {"reads": n, "read_len": 150, "k": k, "m": 2, "gpu": smi or torch.cuda.get_device_name(0), "passes": PASSES}
seq, start, _ = datasets.metagenome_in_memory(n, 150)
stream = torch.cuda.Stream()                                       # the graph's stream: the events bracket its kernels
with cabi.Context(k, 2) as ctx:
    ctx.set_reads(seq, start, max_len=150)
    ctx.stage1()
    g = cabi.Sdbg(k, True, stream=stream.cuda_stream)
    g.from_stage2(ctx)
h = g.finish()
out["edges"] = int(h.size)
last = np.unpackbits(g.array(cabi.SDBG_LAST), bitorder="little")[:h.size].astype(bool)
nodes = torch.from_numpy(np.flatnonzero(last).astype(np.int64)).cuda()
out["nodes"] = int(nodes.numel())
edges = torch.arange(h.size, dtype=torch.int64, device="cuda")
wpt = (2 * k + 31) // 32


def timed(op, x):
    g.query(op, x)                                                 # warm-up
    ts = []
    for _ in range(PASSES):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        r = g.query(op, x)
        b.record(stream)
        b.synchronize()
        ts.append(a.elapsed_time(b) / 1e3)
        del r
    t = sorted(ts)[len(ts) // 2]
    return x.shape[0] / t, t


qps, secs = {}, {}
for name in ["FORWARD", "BACKWARD", "OUTDEGREE", "INDEGREE", "OUTGOING", "INCOMING", "MULTIPLICITY", "REVCOMP", "LABEL"]:
    qps[name], secs[name] = timed(getattr(cabi, "SQ_" + name), edges)
labels = g.label(nodes)[:, :wpt].contiguous()
qps["LABEL_nodes"], secs["LABEL_nodes"] = timed(cabi.SQ_LABEL, nodes)
qps["LOOKUP"], secs["LOOKUP"] = timed(cabi.SQ_LOOKUP, labels)
out["lookup_roundtrip_ok"] = bool(torch.equal(g.lookup(labels), nodes))
os.environ["MGTA_SQ_LV1"] = "0"
qps["LOOKUP_no_lv1"], secs["LOOKUP_no_lv1"] = timed(cabi.SQ_LOOKUP, labels)
out["lookup_no_lv1_same"] = bool(torch.equal(g.lookup(labels), nodes))
del os.environ["MGTA_SQ_LV1"]
g.close()
out["queries_per_s"] = {k_: round(v) for k_, v in qps.items()}
out["median_pass_s"] = {k_: round(v, 6) for k_, v in secs.items()}
print(json.dumps(out))
