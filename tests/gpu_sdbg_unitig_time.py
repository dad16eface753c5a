"""Time of the unitigs of the device SdBG (not a pytest file).
usage: gpu_sdbg_unitig_time.py N_READS [k] [--genome L]   -> one JSON line

The graph of N_READS seeded metagenome reads of 150 bp (m = 2) is built on the device; with --genome L it is instead the
graph of error-free reads tiling one seeded random genome of L bases (m = 1: one unitig of about L edges and its
reverse complement).  mgta_sdbg_unitigs runs once to warm up, then PASSES times between CUDA events on the graph's
stream; the median is reported.  One more pass under torch.profiler gives each kernel's share of the kernel time, and
the copy of the results to host memory is timed on its own."""
import argparse
import json
import os
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import ctypes  # noqa: E402

import numpy as np  # noqa: E402
import torch  # noqa: E402

import datasets  # noqa: E402
from megagta_b200 import cabi  # noqa: E402

PASSES = 3
ap = argparse.ArgumentParser()
ap.add_argument("n_reads", type=int)
ap.add_argument("k", type=int, nargs="?", default=31)
ap.add_argument("--genome", type=int, default=0)
opt = ap.parse_args()
n, k, genome = opt.n_reads, opt.k, opt.genome
m = 1 if genome else 2
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
out = {"reads": n, "read_len": 150, "k": k, "m": m, "genome": genome or None, "gpu": smi or torch.cuda.get_device_name(0),
       "passes": PASSES}
if genome:
    import sdbg_unitig_ref as U
    rd = U.long_genome_reads(genome=genome)
    seq, start, max_len = rd["seq"], rd["start"], rd["max_len"]
    out["reads"] = rd["n_reads"]
else:
    seq, start, _ = datasets.metagenome_in_memory(n, 150)
    max_len = 150
stream = torch.cuda.Stream()                                       # the graph's stream: the events bracket its kernels
with cabi.Context(k, m) as ctx:
    ctx.set_reads(seq, start, max_len=max_len)
    if m > 1:
        ctx.stage1()
    g = cabi.Sdbg(k, True, stream=stream.cuda_stream)
    g.from_stage2(ctx)
h = g.finish()
out["edges"] = int(h.size)
invalid = np.unpackbits(g.array(cabi.SDBG_INVALID), bitorder="little")[:h.size]
out["valid_edges"] = int(h.size - invalid.sum())
n_rows, n_chars = ctypes.c_int64(), ctypes.c_uint64()


def run():
    g._check(g.lib.mgta_sdbg_unitigs(g.h, ctypes.byref(n_rows), ctypes.byref(n_chars)), "mgta_sdbg_unitigs")


run()                                                              # warm-up
ts = []
for _ in range(PASSES):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    run()
    b.record(stream)
    b.synchronize()
    ts.append(a.elapsed_time(b) / 1e3)
out["pass_s"] = [round(t, 6) for t in ts]
out["median_s"] = round(sorted(ts)[len(ts) // 2], 6)
rows, useq = g.unitigs()                                           # computes once more, then copies
rows_b = np.empty_like(rows)
seq_b = np.empty_like(useq)
t2 = time.perf_counter()
g._check(g.lib.mgta_sdbg_unitig_copy(g.h, rows_b.ctypes.data, rows_b.nbytes, seq_b.ctypes.data, seq_b.nbytes), "copy")
t3 = time.perf_counter()
out["copy_to_host_s"] = round(t3 - t2, 6)
out["copy_bytes"] = int(rows_b.nbytes + seq_b.nbytes)
out["same_after_copy"] = bool(np.array_equal(rows_b, rows) and np.array_equal(seq_b, useq))
out["unitigs"] = int(len(rows))
out["chars"] = int(len(useq))
out["longest_unitig_edges"] = int(rows[:, 2].max()) if len(rows) else 0
out["cycles"] = int((rows[:, 5] & cabi.UNITIG_CYCLE).astype(bool).sum())
out["edge_invariant_ok"] = int((rows[:, 2] * np.where(rows[:, 5] & cabi.UNITIG_SELF_RC, 1, 2)).sum()) == out["valid_edges"]
from torch.profiler import ProfilerActivity, profile  # noqa: E402

with profile(activities=[ProfilerActivity.CUDA]) as prof:         # a pass of its own: tracing slows the host
    run()
    torch.cuda.synchronize()
per = {}
for ev in prof.key_averages():
    hit = re.search(r"k_ut_[a-z_]+", ev.key)
    if hit:
        t = getattr(ev, "device_time_total", None)
        per[hit.group(0)] = per.get(hit.group(0), 0.0) + (t if t is not None else ev.cuda_time_total)
tot = sum(per.values())
out["kernel_ms"] = round(tot / 1e3, 3)
out["kernel_share"] = {n_: round(v / tot, 4) for n_, v in sorted(per.items(), key=lambda x: -x[1])} if tot else {}
g.close()
print(json.dumps(out))
