"""bench.py contract on the CPU: the reference arm (`--impl reference`) runs the reference's own CPU CX1 on a bounded
sample and prints one JSON line with the keys the driver reads; the GPU arm's line is checked on the GPU box."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

REQUIRED = ["impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"]


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--sample-reads", "30000",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for k in REQUIRED:
        assert k in line, k
    assert line["impl"] == "reference" and line["metric"] == "SdBG edges/sec" and line["unit"] == "edges/s"
    assert line["value"] > 0 and line["higher_is_better"] is True
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"] and "sample" in line["config"]
    assert line["reads_per_s"] > 0 and len(line["config"]["sample_hashes"]["stream_hash"]) == 16
    assert line["steps"] == line["timed_steps"] == 1


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_dump_outputs_writes_the_step_results_as_float_arrays(read_lib, tmp_path, monkeypatch):
    """--dump-outputs on a graph of the oracle: every array is float32 / float64, equal to what it stands for, and the
    per-bucket digests add up to the parity xsum; a stream larger than the sample is sampled at seeded positions, and a
    shard writes the rows of its own bucket range"""
    import numpy as np
    from oracle import oracle as O
    bench = _bench_module()
    prefix, rd = read_lib("smoke")
    k, m = 31, 2
    res = O.build_graph(rd, k, m)
    wpt = (2 * k + 31) // 32
    last = {"edge_counting": res["counting"], "meta": res["meta"], "totals": res["totals"]}
    dig = bench.bucket_digests(res["stream"], res["meta"], wpt)
    bench.dump_outputs(str(tmp_path), last, res["stream"], dig, 7, 0, 1, (0, 65536))
    got = {f[:-4]: np.load(str(tmp_path / f)) for f in os.listdir(str(tmp_path))}
    assert sorted(got) == ["bucket_table", "edge_counting", "stream_bucket_digest", "stream_sample", "totals"]
    assert all(x.dtype in (np.float32, np.float64) for x in got.values())
    assert sum(os.path.getsize(str(tmp_path / f)) for f in os.listdir(str(tmp_path))) <= 64 << 20
    assert np.array_equal(got["edge_counting"], res["counting"]) and np.array_equal(got["bucket_table"], res["meta"])
    assert np.array_equal(got["totals"], res["totals"])
    d = got["stream_bucket_digest"].astype(np.uint64)
    assert np.array_equal((d[:, 0] << np.uint64(32)) | d[:, 1], dig)
    assert int(dig.sum(dtype=np.uint64)) == bench.bucket_xsum(res["stream"], res["meta"], wpt) != 0
    rec = np.frombuffer(res["stream"], dtype=np.uint8)
    assert len(rec) <= bench.DUMP_STREAM_SAMPLE and np.array_equal(got["stream_sample"], rec)

    monkeypatch.setattr(bench, "DUMP_STREAM_SAMPLE", 4096)
    samples = []
    for i, seed in enumerate((7, 7, 8)):
        d = str(tmp_path / ("sampled%d" % i))
        bench.dump_outputs(d, last, res["stream"], dig, seed, 1, 2, (100, 30000))
        got = {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}
        assert sorted(got) == ["bucket_table", "stream_bucket_digest", "stream_sample", "totals"]      # edge_counting: rank 0
        assert np.array_equal(got["bucket_table"], res["meta"][100:30000]) and len(got["stream_bucket_digest"]) == 29900
        assert got["stream_sample"].dtype == np.float32 and len(got["stream_sample"]) == 2048                # 4096 / world
        pick = np.sort(np.random.default_rng(seed).integers(0, len(rec), size=2048))
        assert np.array_equal(got["stream_sample"], rec[pick])
        samples.append(got["stream_sample"])
    assert np.array_equal(samples[0], samples[1]) and not np.array_equal(samples[0], samples[2])


@pytest.mark.gpu
def test_gpu_arm_dumps_the_same_outputs_on_every_run(tmp_path):
    """same arguments -> same inputs -> the same dumped arrays; --steps is the number of timed steps in the line"""
    import numpy as np
    dumps = []
    for i in range(2):
        d = str(tmp_path / ("run%d" % i))
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--reads-per-gpu", "1000000", "--steps", "2", "--warmup", "1",
                            "--no-cpu-baseline", "--dump-outputs", d], capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == 2 and line["timed_steps"] == {"device": 2, "e2e": 2}
        dumps.append({f: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))})
        assert sum(x.nbytes for x in dumps[-1].values()) <= 64 << 20
        assert dumps[-1]["bucket_table.npy"][:, 0].sum() == line["config"]["edges_per_step"]
        dg = dumps[-1]["stream_bucket_digest.npy"].astype(np.uint64)
        assert "%016x" % int(((dg[:, 0] << np.uint64(32)) | dg[:, 1]).sum(dtype=np.uint64)) == line["config"]["parity"]["xsum"]
    assert sorted(dumps[0]) == sorted(dumps[1]) and len(dumps[0]) == 5
    for f in dumps[0]:
        assert np.array_equal(dumps[0][f], dumps[1][f]), f


@pytest.mark.gpu
def test_gpu_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--reads-per-gpu", "1000000", "--steps", "1", "--warmup", "3",
                        "--sample-reads", "20000"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for k in ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline"]:
        assert k in line, k
    assert line["gpu_launches"] > 0 and line["value"] > 0 and line["e2e"]["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["d2h_bytes_per_step"] > 0
    for k in ["bound", "achieved", "peak", "unit", "frac", "traffic"]:
        assert k in line["roofline"], k
    for k in ["value", "unit", "cores", "kind", "sample"]:
        assert k in line["cpu_baseline"], k
    par = line["config"]["parity"]
    assert par["sample"]["ok"] is True, par["sample"]          # GPU path == reference binary on the shared sample, in this job
    assert len(par["stream_hash"]) == 16 and par["total_size"] == line["config"]["edges_per_step"]
