#!/usr/bin/env python
"""bench.py -- SdBG edges/s of the CX1 reads->SdBG path on N B200s (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W]            our arm (libmgta_cuda.so via its C ABI)
  python bench.py --impl reference [--gpus N] ...                 the reference's CPU CX1 on the host cores

One "step" = one whole buildgraph (stage 1 + stage 2) over the synthetic read set.
  value : inputs resident in HBM, records left in HBM (device work only)
  e2e   : the same call chain from HOST buffers: H2D of the packed reads (+ NCCL broadcast when N>1),
          both stages, D2H of the record stream and the per-bucket table, every step
Workload at N GPUs: 20M x N reads of 150 bp (weak scaling; N=1 is BASELINE.json configs[1]), k=31, m=2.
"""
import argparse
import ctypes
import gc
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "SdBG edges/sec"
UNIT = "edges/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--reads-per-gpu", type=int, default=20_000_000)
    ap.add_argument("--read-len", type=int, default=150)
    ap.add_argument("-k", type=int, default=31)
    ap.add_argument("-m", type=int, default=2)
    ap.add_argument("--sample-reads", type=int, default=0, help="reads in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--seed", type=int, default=20261017)
    ap.add_argument("--genomes-per-gpu", type=int, default=64)
    ap.add_argument("--total-reads", type=int, default=0,
                    help="strong scaling: this many reads in all, split over the GPUs (0 = weak scaling with --reads-per-gpu each)")
    ap.add_argument("--genomes", type=int, default=0, help="genomes of the community (0 = --genomes-per-gpu x GPUs; strong scaling: x total/20M)")
    ap.add_argument("--gen-chunk", type=int, default=1_000_000,
                    help="reads per RNG chunk of the generator (reads per GPU must be a multiple; the read set depends on it)")
    ap.add_argument("--no-hash", action="store_true", help="skip the (untimed) parity hashes of the GPU output")
    ap.add_argument("--full-reference", action="store_true",
                    help="N=1: also build the WHOLE workload with the reference on the host cores (untimed) and compare the hashes")
    ap.add_argument("--phases", action="store_true", help="diagnostic: per-phase host wall times of every rank on stderr (adds syncs)")
    ap.add_argument("--root-upload", action="store_true",
                    help="N>1: rank 0 uploads all reads and broadcasts them (default: every rank uploads its slice, NCCL all-gather)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (N>1: DIR/rank<r>/); "
                         "same arguments -> same inputs, so two builds can be compared output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.total_reads:
        assert a.total_reads % (a.gpus * a.gen_chunk) == 0, "--total-reads must be a multiple of --gen-chunk x GPUs"
        a.reads_per_gpu = a.total_reads // a.gpus
    return a


def n_genomes(a, n_gpus):
    """Weak scaling keeps the per-GPU work fixed: the community grows with the read set (64 genomes per 20M reads, the
    density of BASELINE.json configs[1]), so coverage and the SdBG edges per read stay those of the 1-GPU workload.  With a
    fixed community the edge count saturates as reads are added and edges/s would fall for reasons unrelated to the code."""
    if a.genomes:
        return a.genomes
    if a.total_reads:                                   # strong scaling: the community of the whole read set, whatever N
        return a.genomes_per_gpu * max(1, a.total_reads // 20_000_000)
    return a.genomes_per_gpu * n_gpus


def sample_genomes(a):
    """The CPU sample is drawn from the SAME community at every N (the N = 1 workload's when scaling weakly), so the
    reference arm's value does not wander with N."""
    return a.genomes or (n_genomes(a, 1))


def workload_name(a, n_gpus):
    return "%dM x %d bp synthetic metagenome reads, k=%d, min-count %d" % (
        a.reads_per_gpu * n_gpus // 1_000_000, a.read_len, a.k, a.m)


def bucket_digests(stream, meta, wpt):
    """uint64[65536]: a keyed 64-bit digest (blake2b, salt = bucket) of every non-empty lv1 bucket's bytes of the record
    stream, 0 for an empty bucket."""
    import hashlib
    m = np.asarray(meta, dtype=np.int64)
    sizes = m[:, 0] * 2 + m[:, 2] * 2 + m[:, 1] * 4 * wpt
    out = np.zeros(len(m), dtype=np.uint64)
    off = 0
    mv = memoryview(stream)
    for b in np.nonzero(sizes)[0]:
        n = int(sizes[b])
        out[b] = int.from_bytes(hashlib.blake2b(mv[off:off + n], digest_size=8, salt=int(b).to_bytes(8, "little")).digest(), "little")
        off += n
    assert off == len(stream), "per-bucket table does not add up to the stream"
    return out


def bucket_xsum(stream, meta, wpt):
    """Composable checksum of a shard's record stream: the sum of its bucket_digests (mod 2^64).  Buckets are disjoint
    between shards and batches, so the sums of N shards add up to the 1-GPU value; equal sums <=> equal per-bucket byte
    strings (up to digest collisions)."""
    return int(bucket_digests(stream, meta, wpt).sum(dtype=np.uint64))


DUMP_STREAM_SAMPLE = 8 << 20          # record-stream bytes in a --dump-outputs directory (32 MB as float32)


def dump_outputs(d, last, stream, digests, seed, rank, world, buckets):
    """--dump-outputs: what the last timed step returned -- stage 1's edge_counting, stage 2's per-bucket table and totals --
    and its SdBG record stream (re-emitted from the same graph after the timed region: the timed path leaves the records in
    HBM), as the per-bucket digests (hi, lo 32 bits) of the whole stream and its bytes (a seeded sample when it is larger
    than DUMP_STREAM_SAMPLE / world).  A shard writes the rows of its own bucket range [b0, b1) of the tables, and rank 0
    alone the whole-graph edge_counting, so that the files of all ranks stay at ~35 MB (32 MB sample, 3 MB tables) at any
    N.  float64 holds every integer here exactly."""
    b0, b1 = buckets
    os.makedirs(d, exist_ok=True)
    rec = np.frombuffer(stream, dtype=np.uint8)
    n = DUMP_STREAM_SAMPLE // world
    pick = np.sort(np.random.default_rng(seed).integers(0, len(rec), size=n)) if len(rec) > n else np.arange(len(rec))
    arrays = {"bucket_table": last["meta"][b0:b1], "totals": last["totals"],
              "stream_bucket_digest": np.stack([digests >> np.uint64(32), digests & np.uint64(0xFFFFFFFF)], axis=1)[b0:b1],
              "stream_sample": rec[pick]}
    if rank == 0 and last.get("edge_counting") is not None:              # min-count 1 has no stage 1
        arrays["edge_counting"] = last["edge_counting"]
    for name, x in arrays.items():
        np.save(os.path.join(d, name + ".npy"), x.astype(np.float32 if x.dtype == np.uint8 else np.float64))


# ------------------------------------------------------------------------------------------------ reference arm
def auto_sample(a):
    """Reads of the bounded CPU sample: as many as keep 25 reference runs within the arm's time budget
    (measured: ~5 s per 1M x 150 bp reads on 16 cores, ~3 s on 32)."""
    if a.sample_reads:
        return a.sample_reads
    cores = os.cpu_count() or 1
    return min(a.reads_per_gpu, 2_000_000 if cores <= 16 else 4_000_000)


def write_sample(a, work):
    from megagta_b200 import synth
    n = auto_sample(a)
    prefix = os.path.join(work, "sample")
    synth.packed_metagenome(n, a.read_len, seed=a.seed, bin_prefix=prefix, bin_reads=n, n_genomes=sample_genomes(a), chunk=a.gen_chunk)
    return prefix, n


def time_reference(prefix, a, work, tag, want_hash=False):
    """One run of the unmodified reference buildgraph (oracle/_ref) on all host cores
    -> (seconds, edges, kind, cores, hashes or None)."""
    from oracle import oracle as O
    from megagta_b200 import sdbg_io
    cores = os.cpu_count() or 2
    out = os.path.join(work, "ref_" + tag)
    if O.have_ref():
        t = time.time()
        O.run_ref_buildgraph(prefix, out, a.k, a.m, threads=max(2, cores))
        dt = time.time() - t
        hashes = None
        if want_hash:
            hdr, stream, meta = sdbg_io.canonical(out)
            hashes = {"stream_hash": sdbg_io.stream_hash(stream), "meta_hash": sdbg_io.meta_hash(meta), "stream_bytes": len(stream),
                      "xsum": "%016x" % bucket_xsum(stream, meta, hdr["words_per_tip_label"])}
            del stream
        else:
            hdr, _ = sdbg_io.read_info(out)
        for f in os.listdir(work):
            if f.startswith("ref_" + tag):
                os.remove(os.path.join(work, f))
        return dt, hdr["total_size"], "reference", max(2, cores), hashes
    rd = O.load_read_lib(prefix)                      # fall back to the single-threaded C restatement
    t = time.time()
    res = O.build_graph(rd, a.k, a.m)
    dt = time.time() - t
    hashes = None
    if want_hash:
        wpt = (2 * a.k + 31) // 32
        hashes = {"stream_hash": sdbg_io.stream_hash(res["stream"]), "meta_hash": sdbg_io.meta_hash(res["meta"]),
                  "stream_bytes": len(res["stream"]), "xsum": "%016x" % bucket_xsum(res["stream"], res["meta"], wpt)}
    return dt, int(res["meta"][:, 0].sum()), "port", 1, hashes


def run_reference_arm(a, work):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    prefix, n = write_sample(a, work)
    times, edges, kind, cores, hashes = [], 0, "reference", 1, None
    for i in range(a.warmup + a.steps):
        dt, edges, kind, cores, h = time_reference(prefix, a, work, str(i), want_hash=(i == 0))
        hashes = hashes or h
        if i >= a.warmup:
            times.append(dt)
    ms = 1000.0 * sum(times) / len(times)
    value = edges / (ms / 1000.0)
    sample = "first %d reads of the %d-genome community (%d x %d bp), whole buildgraph, %d threads" % (n, sample_genomes(a), n, a.read_len, cores)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "timed_steps": len(times),
            "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong" if a.total_reads else "weak",
            "vs_baseline": None, "dtype": "u32", "data": "synthetic", "reads_per_s": n / (ms / 1000.0),
            "config": {"workload": workload_name(a, a.gpus), "reads": a.reads_per_gpu * a.gpus, "read_len": a.read_len, "k": a.k,
                       "min_count": a.m, "genomes": n_genomes(a, a.gpus), "sample": sample, "sample_reads": n,
                       "edges_per_step": edges, "sample_hashes": hashes},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample, "reads_per_s": n / (ms / 1000.0)},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ our arm
SAMPLER_CHILD = r"""
import sys, time
uuids = sys.argv[1:]
try:
    import pynvml as n
    n.nvmlInit()
    hs = []
    for i, u in enumerate(uuids):
        try:
            hs.append(n.nvmlDeviceGetHandleByUUID(u.encode()))
        except Exception:
            hs.append(n.nvmlDeviceGetHandleByIndex(i))
    print("max", int(n.nvmlDeviceGetMaxClockInfo(hs[0], n.NVML_CLOCK_SM)), flush=True)
    while True:
        for h in hs:
            sm = int(n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM))
            try:
                mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(h))
            except Exception:
                mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(h))
            print("s", time.time(), sm, mask, flush=True)
        time.sleep(0.2)
except Exception as e:
    print("err", repr(e), flush=True)
"""


class ClockSampler:
    """SM clock + throttle reasons of the job's GPUs during the timed region, sampled 5 times a second by ONE helper
    process of rank 0 through NVML.  It is a separate process on purpose: measured on this path, one nvidia-smi spawn per
    rank every 100 ms slowed the 2-GPU step from 246 to 304 ms, and an in-process NVML thread left 17-34 ms of host gaps in
    stage 2 (1-2 ms without it) -- the queries serialise with the process's own driver calls.  nvidia-smi (one query
    before and one after) is the fallback when the binding is missing."""
    REASONS = [(0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap")]

    def __init__(self, devs):
        import torch
        self.devs, self.rows, self.max_mhz, self.source = list(devs), [], None, "nvml (helper process)"
        uuids = []
        for d in self.devs:
            try:
                uuids.append("GPU-" + str(torch.cuda.get_device_properties(d).uuid))
            except Exception:
                uuids.append("")
        self.t0 = self.t1 = None
        try:
            self.proc = subprocess.Popen([sys.executable, "-c", SAMPLER_CHILD] + uuids, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                                         text=True)
        except Exception:
            self.proc = None

    def start(self):
        self.t0 = time.time()

    def join(self):
        self.t1 = time.time()
        if self.proc:
            self.proc.terminate()
            try:
                out = self.proc.communicate(timeout=5)[0]
            except Exception:
                out = ""
            for line in out.splitlines():
                f = line.split()
                if f and f[0] == "max":
                    self.max_mhz = int(f[1])
                elif f and f[0] == "s" and self.t0 <= float(f[1]) <= self.t1:
                    self.rows.append((int(f[2]), int(f[3])))
        if not self.rows:
            self.sample_smi()

    stop_flag = False

    def sample_smi(self):
        self.source = "nvidia-smi (after the timed region)"
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            o = subprocess.run(["nvidia-smi", "-i", ",".join(str(d) for d in self.devs), "--query-gpu=" + q,
                                "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout.strip()
        except Exception:
            o = ""
        for line in o.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) >= 6 and f[0].isdigit():
                if f[1].isdigit():
                    self.max_mhz = int(f[1])
                mask = sum(bit for (bit, _), v in zip(self.REASONS, f[2:6]) if v.lower().startswith("active"))
                self.rows.append((int(f[0]), mask))

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0, "source": self.source}
        sm = sorted(r[0] for r in self.rows)
        reasons = [name for bit, name in self.REASONS if any(r[1] & bit for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(self.rows), "gpus_sampled": len(self.devs), "source": self.source}


class DevBuf:
    def __init__(self, ptr, nbytes, typestr="<i4", itemsize=4):
        self.__cuda_array_interface__ = {"shape": (nbytes // itemsize,), "typestr": typestr, "data": (ptr, False), "version": 3}


def main():
    a = parse()
    work = tempfile.mkdtemp(prefix="mgta_bench_")          # the sample read library and the reference's files
    try:
        return run_reference_arm(a, work) if a.impl == "reference" else run_gpu_arm(a, work)
    finally:
        shutil.rmtree(work, ignore_errors=True)


def run_gpu_arm(a, work):

    import torch
    import torch.distributed as dist
    from megagta_b200 import cabi, shards, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    n_gpus = world
    n_reads = a.reads_per_gpu * n_gpus
    L = a.read_len

    # ---- synthetic reads (rank 0 only; the other ranks receive them over NVLink)
    sample_prefix, sample_n = os.path.join(work, "sample"), auto_sample(a)
    n_words = n_reads * L // 16 + 1
    # N = 1 (or --root-upload): rank 0 holds all reads, uploads them and broadcasts.  N > 1: every rank holds ITS slice of the
    # read set in pinned host memory (as if it had read its part of the .bin file), uploads it over its own PCIe link into
    # place in the full device buffer, and one NCCL all-gather over NVLink completes the buffers on every GPU.
    sharded_upload = world > 1 and not a.root_upload
    per_words = a.reads_per_gpu * L // 16                      # words of one shard's slice (reads_per_gpu * L % 16 == 0)
    assert not sharded_upload or (a.reads_per_gpu * L) % 16 == 0 and a.reads_per_gpu % a.gen_chunk == 0
    # Pinned staging buffers should live on the NUMA node the GPU hangs off (first touch follows the thread): bind this
    # process to the GPU's CPUs (NVML) while it allocates and runs the GPU arm; the CPU baseline gets all cores back.
    full_affinity = os.sched_getaffinity(0)
    near_count = len(full_affinity)
    try:
        import pynvml
        pynvml.nvmlInit()
        try:
            h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(torch.cuda.get_device_properties(local).uuid)).encode())
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64 + 16)
        near = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1} & full_affinity
        if len(near) >= 2:
            os.sched_setaffinity(0, near)
            near_count = len(near)
    except Exception:
        pass
    t0 = time.time()
    if sharded_upload:
        seq, start = synth.packed_metagenome(a.reads_per_gpu, L, seed=a.seed, first_read=rank * a.reads_per_gpu, n_genomes=n_genomes(a, world),
                                             bin_prefix=sample_prefix if rank == 0 else None, bin_reads=sample_n if rank == 0 else 0,
                                             procs=max(1, (os.cpu_count() or 8) // world), chunk=a.gen_chunk)
        seq_pin = torch.from_numpy(seq[:per_words].view(np.int32)).pin_memory()
        start_pin = torch.from_numpy((start[:a.reads_per_gpu] + np.uint64(rank * a.reads_per_gpu * L)).view(np.int64)).pin_memory()
        del seq, start
    elif rank == 0:
        seq, start = synth.packed_metagenome(n_reads, L, seed=a.seed, bin_prefix=sample_prefix,
                                             bin_reads=n_reads if (a.full_reference and world == 1) else sample_n, n_genomes=n_genomes(a, world),
                                             chunk=a.gen_chunk)
        seq_pin = torch.from_numpy(seq).pin_memory()
        start_pin = torch.from_numpy(start.view(np.int64)).pin_memory()
        del seq, start
    gen_s = time.time() - t0
    stream = torch.cuda.Stream(device=dev)
    ctx = cabi.Context(a.k, a.m, device=local, rank=rank, world=world, stream=stream.cuda_stream)

    def load_reads():
        """host -> HBM (+ all-gather / broadcast over NVLink).  Returns H2D bytes of this rank."""
        h2d = 0
        if sharded_upload:
            ctx.alloc_reads(n_words, n_reads, n_reads, n_reads * L, L)
            (sp, sb), (tp, tb) = ctx.reads_device_buffers()
            d_seq = torch.as_tensor(DevBuf(sp, world * per_words * 4), device=dev)             # the last (+1) word stays zero
            d_start = torch.as_tensor(DevBuf(tp, n_reads * 8, "<i8", 8), device=dev)
            d_seq[rank * per_words:(rank + 1) * per_words].copy_(seq_pin, non_blocking=True)
            d_start[rank * a.reads_per_gpu:(rank + 1) * a.reads_per_gpu].copy_(start_pin, non_blocking=True)
            dist.all_gather_into_tensor(d_seq, d_seq[rank * per_words:(rank + 1) * per_words])
            dist.all_gather_into_tensor(d_start, d_start[rank * a.reads_per_gpu:(rank + 1) * a.reads_per_gpu])
            torch.as_tensor(DevBuf(tp + n_reads * 8, 8, "<i8", 8), device=dev).fill_(n_reads * L)   # start_idx[n_reads]
            torch.as_tensor(DevBuf(sp + world * per_words * 4, 4), device=dev).fill_(0)             # the spare last word
            h2d = per_words * 4 + a.reads_per_gpu * 8
        elif rank == 0:
            # pinned buffers that outlive the step: the asynchronous upload hides behind the stage-1 extraction
            ctx._check(ctx.lib.mgta_set_reads_async(ctx.h, seq_pin.data_ptr(), n_words, start_pin.data_ptr(), n_reads, n_reads, L),
                       "mgta_set_reads_async")
            ctx.n_short, ctx.max_len = n_reads, L
            h2d = n_words * 4 + (n_reads + 1) * 8
        else:
            ctx.alloc_reads(n_words, n_reads, n_reads, n_reads * L, L)
        if world > 1 and not sharded_upload:
            (sp, sb), (tp, tb) = ctx.reads_device_buffers()
            dist.broadcast(torch.as_tensor(DevBuf(sp, sb), device=dev), 0)
            dist.broadcast(torch.as_tensor(DevBuf(tp, tb), device=dev), 0)
        return h2d

    phases = {}

    def mark(name, t0):
        if not a.phases:
            return t0
        torch.cuda.synchronize()
        phases.setdefault(name, []).append(round((time.time() - t0) * 1000, 1))
        return time.time()

    comm = shards.TorchComm(ctx, rank, world, dist, dev) if world > 1 else None
    last = {}                                  # what the latest step returned (--dump-outputs)

    def step(e2e):
        """-> (edges of this shard, h2d bytes, d2h bytes).  N > 1: the library walks the sharded protocol
        (mgta_sharded_begin / _step), TorchComm runs the collectives it asks for over NCCL."""
        t = time.time()
        h2d = load_reads() if e2e else 0
        t = mark("load", t)
        d2h = 0
        if a.m > 1:
            last["edge_counting"] = ctx.sharded(1, comm) if world > 1 else ctx.stage1()
            t = mark("stage1", t)
        collect = "count" if e2e else False
        nbytes, meta, totals = ctx.sharded(2, comm, collect=collect) if world > 1 else ctx.stage2(collect=collect)
        last["meta"], last["totals"] = meta, totals
        if e2e:
            d2h = nbytes + meta[slice(*ctx.shard_range())].nbytes
        mark("stage2", t)
        return ctx.stats(2)["n_edges"], h2d, d2h

    def timed(fn, reps):
        """barrier + sync, CUDA events on the launching stream, max over ranks -> ms per rep"""
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        gc.collect()
        gc.disable()                                 # a collector pause on one rank stalls every rank at the next collective
        e0.record(stream)
        outs = [fn() for _ in range(reps)]
        e1.record(stream)
        gc.enable()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / reps, outs

    sampler = ClockSampler(range(world)) if rank == 0 else None         # rank 0 watches all GPUs of the job (one node);
    if os.environ.get("MGTA_BENCH_SAMPLER") == "off":                   # started here so that it is up before the timed region
        sampler = None                                                  # (off: diagnostic only)
    with torch.cuda.stream(stream):
        load_reads()
        for _ in range(a.warmup):
            step(False)
        if sampler:
            sampler.start()
        ms_dev, outs = timed(lambda: step(False), a.steps)
        st1, st2 = ctx.stats(1), ctx.stats(2)
        step(True)      # untimed: the first end-to-end call allocates the library's pinned output staging (cudaHostAlloc)
        ms_e2e, outs_e2e = timed(lambda: step(True), a.steps)
        if sampler:
            sampler.stop_flag = True
            sampler.join()

    # ---- parity evidence, outside every timed region: hashes of the records the last step's graph emits
    parity = {}
    wpt = (2 * a.k + 31) // 32
    if not a.no_hash or a.dump_outputs:
        with torch.cuda.stream(stream):
            h_stream, h_meta, h_totals = ctx.sharded(2, comm, collect=True) if world > 1 else ctx.stage2(collect=True)
        assert np.array_equal(h_meta, last["meta"]) and np.array_equal(h_totals, last["totals"]), \
            "stage 2 emitted again differs from the last timed step"
        digests = bucket_digests(h_stream, h_meta, wpt)
        if a.dump_outputs:
            dump_outputs(a.dump_outputs if world == 1 else os.path.join(a.dump_outputs, "rank%d" % rank), last, h_stream, digests,
                         a.seed, rank, world, ctx.shard_range())
    if not a.no_hash:
        xs = int(digests.sum(dtype=np.uint64))
        part = torch.tensor([xs & 0xFFFFFFFF, xs >> 32, len(h_stream), int(h_meta[:, 0].sum()), int(h_meta[:, 1].sum())], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(part, op=dist.ReduceOp.SUM)
        pl = [int(x) for x in part.tolist()]
        parity = {"xsum": "%016x" % ((pl[0] + (pl[1] << 32)) & 0xFFFFFFFFFFFFFFFF), "stream_bytes": pl[2], "total_size": pl[3],
                  "num_tips": pl[4],
                  "xsum_def": "sum over lv1 buckets of blake2b-64(bucket bytes, salt = bucket) mod 2^64: composable over shards"}
        if world == 1:
            from megagta_b200 import sdbg_io
            parity["stream_hash"] = sdbg_io.stream_hash(h_stream)
            parity["meta_hash"] = sdbg_io.meta_hash(h_meta)
        del h_stream

    def total(x):
        t = torch.tensor([float(x)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # the reference's own stage-2 item count (its lv1 histogram), for the SURVEY-model figure; outside every timed region
    ref_s2_items = 0
    if world == 1:
        try:
            ref_s2_items = int(ctx.histogram(2).sum())
        except Exception:
            ref_s2_items = 0
    if a.phases:
        sys.stderr.write("rank %d phases(ms) %s\n" % (rank, json.dumps(phases)))
    edges = total(outs[-1][0])
    h2d = total(outs_e2e[-1][1])
    d2h = total(outs_e2e[-1][2])
    launches = total(st1["n_launches"] + st2["n_launches"]) * a.steps

    if rank == 0:
        peaks = {}
        pk_src = "fallback"
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
            pk_src = "measured"
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        # per-kernel algorithmic bytes (DESIGN.md section 5): what each kernel must read + write once
        seq_bytes = n_words * 4
        kern = []
        n1, iw1, rows = st1["n_items"], st1["item_words"], st1["n_edges"]
        row_bytes = (st1["key_words"] + 1) * 4
        if n1:
            sharded = world > 1
            kern.append(("s1.k_edge_part", st1["ms_extract"], (seq_bytes // world if sharded else seq_bytes * max(1, st1["n_batches"])) + n1 * iw1 * 4))
            kern.append(("s1.k_split", st1["ms_partition"], (4 if sharded else 2) * n1 * iw1 * 4))
            kern.append(("s1.k_count", st1["ms_sort_emit"], n1 * iw1 * 4 + rows * row_bytes))
        n2, iw2 = st2["n_items"], st2["item_words"]
        nops, ntip = st2.get("n_node_ops", 0), st2.get("n_tip_items", 0)
        if nops:
            # node pass (k_node_part + k_split + k_node_count): edge rows in, ops written, split, counted; tip rows out
            iwn = (2 * a.k + 31) // 32 + 1
            kern.append(("s2.node_pass", st2["ms_nodes"], rows * row_bytes + 4 * nops * iwn * 4 + ntip * iw2 * 4))
        if n2:
            kern.append(("s2.k_item_part", st2["ms_extract"], (rows * row_bytes + ntip * iw2 * 4) * max(1, st2["n_batches"]) + n2 * iw2 * 4))
            kern.append(("s2.k_split", st2["ms_partition"], 2 * n2 * iw2 * 4))
            kern.append(("s2.k_sort_emit", st2["ms_sort_emit"], n2 * iw2 * 4 + st2["out_bytes"]))
        kern.sort(key=lambda x: -x[1])
        top = kern[0]
        ach = top[2] / (top[1] / 1000.0) / 1e9 if top[1] > 0 else 0.0
        step_bytes = sum(k[2] for k in kern)
        traffic = None                                 # DRAM bytes of the kernel from the committed ncu capture, same configuration only
        try:                                           # profiles/traffic.json is generated by tools/ncu_traffic.py, never by hand
            tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            c = tr["config"]
            if (n_gpus == c["n_gpus"] and n_reads == c["reads"] and L == c["read_len"] and a.k == c["k"] and a.m == c["min_count"]
                    and n1 == tr["s1_items"] and n2 == tr["s2_items"] and top[0] in tr["kernels"]):
                e = tr["kernels"][top[0]]
                traffic = e["dram_bytes_read"] + e["dram_bytes_write"]
        except Exception:
            traffic = None
        roofline = {"bound": "hbm", "kernel": top[0], "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": traffic, "peak_source": pk_src, "algorithmic_bytes_per_launch": top[2],
                    "step_algorithmic_bytes": step_bytes, "step_frac": step_bytes / (ms_dev / 1000.0) / 1e9 / peak / n_gpus,
                    "kernels": [{"name": k[0], "ms": k[1], "bytes": k[2], "gbs": (k[2] / (k[1] / 1000.0) / 1e9 if k[1] > 0 else 0.0)}
                                for k in kern]}
        # What binds the dominant kernel is the instruction issue rate, not HBM (DESIGN.md 6.1): warp instructions of the
        # kernel from the same ncu capture as `traffic` / (SMs x 4 issue slots x SM clock) = the time at 100 % issue
        try:
            if traffic is not None and e.get("warp_instructions"):
                clk = sampler.summary() if sampler else None
                sm_mhz = float((clk or {}).get("sm_mhz") or peaks.get("sm_max_mhz") or 1965.0)
                n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
                floor_ms = e["warp_instructions"] / (n_sm * 4.0 * sm_mhz * 1e3)
                roofline["issue"] = {"warp_instructions": e["warp_instructions"], "floor_ms": floor_ms,
                                     "frac": floor_ms / top[1] if top[1] > 0 else None,
                                     "per_item": e["warp_instructions"] * 32.0 / n1 if n1 else None}
        except Exception:
            pass
        # SURVEY 8(d) model: bytes an 8-bit LSD over all key bits below the bucket prefix would move for the REFERENCE's
        # item counts (320 B / 192 B per item at k=31); reported beside the honest per-kernel figure, never instead of it
        def model_bytes_per_item(stage):
            W = -(-(2 * (a.k - 1) + 6) // 32) if stage == 1 else -(-(2 * a.k + 4) // 32)
            bits = 2 * (a.k - 1) + 6 if stage == 1 else 2 * a.k + 4
            P = -(-(bits - 16) // 8)
            return (4 * W + (8 if stage == 1 else 0)) * (2 + 2 * P)
        ref_i1 = n_reads * (L - a.k + 4) if a.m > 1 else 0
        # SURVEY 8(d)'s named counter: DRAM bytes the sort kernel moves per SdBG edge (from the same ncu capture)
        roofline["sort_bytes_per_edge"] = traffic / edges if traffic and edges else None
        roofline["model"] = {"s1_items_ref": ref_i1, "s2_items_ref": ref_s2_items, "bytes_per_item": [model_bytes_per_item(1), model_bytes_per_item(2)],
                             "frac": ((ref_i1 * model_bytes_per_item(1) + ref_s2_items * model_bytes_per_item(2)) / (ms_dev / 1000.0) / 1e9 / peak / n_gpus)
                             if ref_s2_items else None}
        # bytes the reference's LSD model would move per item (SURVEY 8(d)) vs what the kernels above move
        cpu_baseline = None
        try:
            os.sched_setaffinity(0, full_affinity)                 # the reference arm uses every host core
        except Exception:
            pass
        if n_gpus == 1 and not a.no_cpu_baseline:
            if a.full_reference:                                   # the sample library is the first sample_n records of the full one
                full_prefix = os.path.join(work, "full")
                os.rename(sample_prefix + ".bin", full_prefix + ".bin")
                with open(full_prefix + ".lib_info", "w") as f:
                    f.write("%d %d\nsynthetic\n0 %d %d se\n" % (n_reads * L, n_reads, n_reads - 1, L))
                rec = 4 * (1 + (L + 15) // 16)
                with open(full_prefix + ".bin", "rb") as fi, open(sample_prefix + ".bin", "wb") as fo:
                    fo.write(fi.read(sample_n * rec))
                with open(sample_prefix + ".lib_info", "w") as f:
                    f.write("%d %d\nsynthetic\n0 %d %d se\n" % (sample_n * L, sample_n, sample_n - 1, L))
            dt, e, kind, cores, ref_h = time_reference(sample_prefix, a, work, "cpu", want_hash=not a.no_hash)
            cpu_baseline = {"value": e / dt, "unit": UNIT, "cores": cores, "kind": kind, "seconds": dt, "reads_per_s": sample_n / dt,
                            "sample": "first %d reads of the workload (%d x %d bp), whole buildgraph" % (sample_n, sample_n, L)}
            if not a.no_hash:
                # the GPU path on the SAME sample the reference just built: hashes must agree (cx1_read2sdbg_s2.cpp:742-835 output)
                from megagta_b200 import sdbg_io
                ws = (sample_n * L + 15) // 16
                with torch.cuda.stream(stream), cabi.Context(a.k, a.m, device=local, stream=stream.cuda_stream) as c2:
                    c2.set_reads(seq_pin.numpy().view(np.uint32)[:ws], start_pin.numpy().view(np.uint64)[:sample_n + 1], max_len=L)
                    if a.m > 1:
                        c2.stage1()
                    s2_stream, s2_meta, _ = c2.stage2()
                got = {"stream_hash": sdbg_io.stream_hash(s2_stream), "meta_hash": sdbg_io.meta_hash(s2_meta), "stream_bytes": len(s2_stream),
                       "xsum": "%016x" % bucket_xsum(s2_stream, s2_meta, wpt)}
                parity["sample"] = {"reads": sample_n, "gpu": got, "reference": ref_h, "ok": got == ref_h}
                del s2_stream
            if a.full_reference:
                dtf, ef, kindf, coresf, full_h = time_reference(full_prefix, a, work, "full", want_hash=True)
                mine = {k: parity.get(k) for k in ("stream_hash", "meta_hash", "stream_bytes", "xsum")}
                parity["full"] = {"reads": n_reads, "gpu": mine, "reference": full_h, "ok": mine == full_h, "reference_seconds": dtf,
                                  "reference_cores": coresf, "reference_edges_per_s": ef / dtf, "reference_reads_per_s": n_reads / dtf}
        line = {"metric": METRIC, "value": edges / (ms_dev / 1000.0), "unit": UNIT, "n_gpus": n_gpus, "steps": a.steps,
                "timed_steps": {"device": len(outs), "e2e": len(outs_e2e)},
                "warmup": a.warmup, "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "strong" if a.total_reads else "weak",
                "vs_baseline": None, "dtype": "u32", "data": "synthetic", "reads_per_s": n_reads / (ms_dev / 1000.0),
                "config": {"workload": workload_name(a, n_gpus), "reads": n_reads, "read_len": L, "k": a.k, "min_count": a.m,
                           "parity": parity,
                           "genomes": n_genomes(a, n_gpus),
                           "edges_per_step": edges, "s1_items": total_items(st1, world, dist, dev, torch),
                           "s2_items": total_items(st2, world, dist, dev, torch),
                           "l2": "inputs larger than L2 (item arrays are GBs per step); no explicit flush",
                           "sharding": "contiguous lv1-bucket ranges, %d shard(s)" % world,
                           "stage1": ("one shard" if world == 1
                                      else "scan-sharded: each shard scans 1/N of the reads, NCCL all-to-all of the items by hash owner"),
                           "upload": ("rank 0 H2D" + (" + NCCL broadcast" if world > 1 else "") if not sharded_upload
                                      else "every rank H2D of its slice + NCCL all-gather"),
                           "cpu_affinity": "GPU-local CPUs (%d of %d) for the GPU arm" % (near_count, len(full_affinity)),
                           "gen_seconds": gen_s},
                "e2e": {"value": edges / (ms_e2e / 1000.0), "unit": UNIT, "ms_per_step": ms_e2e,
                        "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
                "gpu_launches": int(launches), "clocks": sampler.summary() if sampler else None, "roofline": roofline,
                "stage_ms": {"s1": st1["ms_total"], "s2": st2["ms_total"]},
                "stats": {"s1": st1, "s2": st2}}
        if cpu_baseline:
            line["cpu_baseline"] = cpu_baseline
        print(json.dumps(line), flush=True)
    else:
        total_items(st1, world, dist, dev, torch)
        total_items(st2, world, dist, dev, torch)
    ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def total_items(st, world, dist, dev, torch):
    t = torch.tensor([float(st["n_items"])], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


if __name__ == "__main__":
    main()
