"""Navigation queries on the device SdBG (include/mgta_sdbg_query.h, megagta_b200/csrc/sdbg_query.cu) against the numpy
restatement (tests/sdbg_query_ref.py), every op over every edge, on the graphs of the index tests (test_sdbg_index.py)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import sdbg_query_ref as R
from oracle import oracle as O
from oracle import sdbg_oracle as SO

CASES = [("tiny", 25, 2), ("smoke", 31, 2), ("smoke", 13, 2), ("smoke", 61, 2), ("adversarial", 31, 2), ("adversarial", 21, 1),
         ("xander", 29, 1), ("xander", 33, 1)]
_REF = {}


def restated(rd, ds, k, m, need_mult):
    key = (ds, k, m, need_mult)
    if key not in _REF:
        res = O.build_graph(rd, k, m)
        _REF[key] = R.Restated(SO.build(res["stream"], np.asarray(res["meta"]), k, bool(need_mult)), k)
    return _REF[key]


def lookup_queries(ref, seed):
    """every node label, their reverse complements and seeded random k-mers"""
    lab = R.unpack_chars(R.pack_chars(ref.lab[ref.last_pos]), ref.k)
    rng = np.random.default_rng(seed)
    rnd = rng.integers(0, 4, size=(max(1000, len(lab) // 4), ref.k), dtype=np.uint8)
    return R.pack_chars(np.concatenate([lab, (3 - lab)[:, ::-1], rnd]))


def check_all_ops(g, ref, need_mult, seed=0):
    from megagta_b200 import cabi
    edges = np.arange(ref.size, dtype=np.int64)
    for op in R.EDGE_OPS:
        if op == R.SQ_MULTIPLICITY and not need_mult:
            continue
        got = g.query(op, edges)
        want = ref.run(op, edges)
        if op == R.SQ_LABEL:
            want = want.astype(np.uint32)
        assert np.array_equal(got.reshape(want.shape), want), (op, np.flatnonzero((got.reshape(want.shape) != want).reshape(len(edges), -1).any(axis=1))[:10])
    q = lookup_queries(ref, seed)
    assert np.array_equal(g.query(cabi.SQ_LOOKUP, q), ref.run(R.SQ_LOOKUP, q))


def build(cabi, rd, k, m, need_mult, how, tmp_path=None):
    g = cabi.Sdbg(k, bool(need_mult))
    if how == "files":
        prefix = str(tmp_path / "ref")
        g.from_files(prefix)
    else:
        with cabi.Context(k, m, device=0) as ctx:
            ctx.set_reads(rd["seq"], rd["start"], max_len=rd["max_len"])
            if m > 1:
                ctx.stage1()
            if how == "device":
                g.from_stage2(ctx)
            else:
                stream, meta, _ = ctx.stage2()
                byts = meta[:, 0] * 2 + meta[:, 2] * 2 + meta[:, 1] * 4 * ((2 * k + 31) // 32)
                off = np.concatenate([[0], np.cumsum(byts)])
                for a, b in zip([0, 1, 777, 40001], [1, 777, 40001, 65536]):
                    g.append(a, b, stream[int(off[a]):int(off[b])], meta[a:b])
    g.finish()
    return g


@pytest.mark.gpu
@pytest.mark.parametrize("ds,k,m", CASES)
@pytest.mark.parametrize("need_mult,how", [(1, "device"), (0, "device"), (1, "host")])
def test_gpu_every_op_on_every_edge_equals_the_restatement(read_lib, ds, k, m, need_mult, how):
    from megagta_b200 import cabi
    _, rd = read_lib(ds)
    ref = restated(rd, ds, k, m, need_mult)
    with build(cabi, rd, k, m, need_mult, how) as g:
        assert g.header().size == ref.size
        check_all_ops(g, ref, need_mult, seed=k)


@pytest.mark.gpu
@pytest.mark.parametrize("need_mult", [1, 0])
def test_gpu_queries_on_the_files_of_the_reference_buildgraph(read_lib, tmp_path, need_mult):
    from megagta_b200 import cabi
    if not O.have_ref():
        pytest.skip("oracle/_ref/megagta_ref not built")
    prefix, rd = read_lib("smoke")
    k, m = 31, 2
    O.run_ref_buildgraph(prefix, str(tmp_path / "ref"), k, m)
    ref = restated(rd, "smoke", k, m, need_mult)
    with build(cabi, rd, k, m, need_mult, "files", tmp_path) as g:
        check_all_ops(g, ref, need_mult)


@pytest.mark.gpu
def test_gpu_largest_index_dataset(read_lib):
    from megagta_b200 import cabi
    _, rd = read_lib("meta200k")
    ref = restated(rd, "meta200k", 31, 2, 1)
    with build(cabi, rd, 31, 2, 1, "device") as g:
        check_all_ops(g, ref, 1)


@pytest.mark.gpu
def test_gpu_host_device_numpy_torch_and_chunks_agree(read_lib, monkeypatch):
    import torch
    from megagta_b200 import cabi
    _, rd = read_lib("adversarial")
    k, m = 31, 2
    ref = restated(rd, "adversarial", k, m, 1)
    rng = np.random.default_rng(3)
    edges = rng.integers(0, ref.size, size=50_000).astype(np.int64)
    kmers = lookup_queries(ref, 4)
    with build(cabi, rd, k, m, 1, "device") as g:
        for op in R.EDGE_OPS + [R.SQ_LOOKUP]:
            x = kmers if op == R.SQ_LOOKUP else edges
            host = g.query(op, x)
            dev = g.query(op, torch.from_numpy(x.view(np.int32) if op == R.SQ_LOOKUP else x).cuda())
            assert dev.is_cuda
            assert np.array_equal(dev.cpu().numpy().view(host.dtype).reshape(host.shape), host), op
            # device input, host output and host input, device output, straight through the C ABI
            xd = torch.from_numpy(x.view(np.int32) if op == R.SQ_LOOKUP else x).cuda()
            out_h = np.empty_like(host)
            torch.cuda.synchronize()
            assert g.lib.mgta_sdbg_query(g.h, op, xd.data_ptr(), len(x), out_h.ctypes.data, out_h.nbytes) == 0
            assert np.array_equal(out_h, host), op
            out_d = torch.empty(host.nbytes, dtype=torch.uint8, device="cuda")
            assert g.lib.mgta_sdbg_query(g.h, op, x.ctypes.data, len(x), out_d.data_ptr(), host.nbytes) == 0
            assert np.array_equal(out_d.cpu().numpy().view(host.dtype).reshape(host.shape), host), op
            monkeypatch.setenv("MGTA_SQ_CHUNK_ROWS", "777")       # many staging chunks give the same rows
            assert np.array_equal(g.query(op, x), host), op
            monkeypatch.delenv("MGTA_SQ_CHUNK_ROWS")
        monkeypatch.setenv("MGTA_SQ_LV1", "0")                     # LOOKUP from the f blocks instead of the lv1 bucket
        assert np.array_equal(g.lookup(kmers), ref.run(R.SQ_LOOKUP, kmers))
        monkeypatch.delenv("MGTA_SQ_LV1")
        assert len(g.forward(np.zeros(0, np.int64))) == 0         # n = 0 succeeds


@pytest.mark.gpu
def test_gpu_error_paths_leave_the_graph_usable(read_lib):
    from megagta_b200 import cabi
    _, rd = read_lib("tiny")
    k, m = 25, 2
    ref = restated(rd, "tiny", k, m, 0)
    ok = np.arange(ref.size, dtype=np.int64)
    with cabi.Sdbg(k, True) as g:                                  # before finish
        with pytest.raises(cabi.MgtaError, match="finish"):
            g.forward(ok[:3])
    with build(cabi, rd, k, m, 0, "device") as g:
        with pytest.raises(cabi.MgtaError, match="MULTIPLICITY"):
            g.multiplicity(ok[:3])
        for bad, row in [(np.array([0, 5, ref.size, -1], np.int64), 2), (np.array([-7], np.int64), 0)]:
            with pytest.raises(cabi.MgtaError, match="row %d:" % row):
                g.backward(bad)
            assert np.array_equal(g.forward(ok), ref.fwd)
        out = np.empty(4, np.int64)
        lib = g.lib
        assert lib.mgta_sdbg_query(g.h, 99, ok.ctypes.data, 4, out.ctypes.data, out.nbytes) == -1
        assert b"unknown op" in lib.mgta_sdbg_last_error(g.h)
        assert lib.mgta_sdbg_query(g.h, cabi.SQ_FORWARD, ok.ctypes.data, 5, out.ctypes.data, out.nbytes) == -1
        assert lib.mgta_sdbg_query(g.h, cabi.SQ_FORWARD, ok.ctypes.data, 4, out.ctypes.data, out.nbytes) == 0
        assert np.array_equal(out, ref.fwd[:4])
        a, b = ctypes.c_uint64(), ctypes.c_uint64()
        assert lib.mgta_sdbg_query_row_bytes(g.h, cabi.SQ_LABEL, ctypes.byref(a), ctypes.byref(b)) == 0
        assert (a.value, b.value) == (8, 4 * (ref.wpt + 1))


@pytest.mark.gpu
def test_gpu_query_timing_script_runs(tmp_path):
    script = os.path.join(os.path.dirname(os.path.abspath(__file__)), "gpu_sdbg_query_time.py")
    r = subprocess.run(["python3", script, "20000", "31"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    import json
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["edges"] > 0 and line["lookup_roundtrip_ok"] and line["queries_per_s"]["FORWARD"] > 0
