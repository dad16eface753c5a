"""Unitigs of the device SdBG (include/mgta_sdbg_unitig.h, megagta_b200/csrc/sdbg_unitig.cu) against the restated rows
(tests/sdbg_unitig_ref.py), byte for byte, on the graphs of the query tests and on a long unitig, a long cycle and short
cycles, at several ruler strides."""
import json
import os
import subprocess

import numpy as np
import pytest

import sdbg_query_ref as R
import sdbg_unitig_ref as U
from oracle import oracle as O
from oracle import sdbg_oracle as SO
from test_gpu_sdbg_query import CASES, build, restated

SHAPES = {"long": (U.long_genome_reads, 31), "circular": (U.circular_genome_reads, 31), "tandem": (U.tandem_reads, 21)}


def check_unitigs(g, ref):
    rows, seq = g.unitigs()
    want_rows, want_seq = U.restated_unitigs(ref)
    assert np.array_equal(rows, want_rows), np.flatnonzero((rows != want_rows).any(axis=1))[:10] if rows.shape == want_rows.shape else rows.shape
    assert np.array_equal(seq, want_seq)
    assert U.edge_invariant(rows) == int((~ref.invalid).sum())
    return rows, seq


@pytest.mark.gpu
@pytest.mark.parametrize("ds,k,m", CASES)
@pytest.mark.parametrize("need_mult,how", [(1, "device"), (0, "device"), (1, "host")])
def test_gpu_unitigs_equal_the_restatement(read_lib, ds, k, m, need_mult, how):
    from megagta_b200 import cabi
    _, rd = read_lib(ds)
    ref = restated(rd, ds, k, m, need_mult)
    with build(cabi, rd, k, m, need_mult, how) as g:
        rows, _ = check_unitigs(g, ref)
        assert (rows[:, 4] >= 0).all() if need_mult else (rows[:, 4] == -1).all()


@pytest.mark.gpu
def test_gpu_unitigs_on_the_files_of_the_reference_buildgraph(read_lib, tmp_path):
    from megagta_b200 import cabi
    if not O.have_ref():
        pytest.skip("oracle/_ref/megagta_ref not built")
    prefix, rd = read_lib("smoke")
    k, m = 31, 2
    O.run_ref_buildgraph(prefix, str(tmp_path / "ref"), k, m)
    with build(cabi, rd, k, m, 1, "files", tmp_path) as g:
        check_unitigs(g, restated(rd, "smoke", k, m, 1))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", sorted(SHAPES))
def test_gpu_hard_shapes_at_every_ruler_stride(shape, monkeypatch):
    from megagta_b200 import cabi
    gen, k = SHAPES[shape]
    rd = gen()
    res = O.build_graph(rd, k, 1)
    ref = R.Restated(SO.build(res["stream"], np.asarray(res["meta"]), k, True), k)
    with build(cabi, rd, k, 1, 1, "device") as g:
        first = None
        for stride in ("1", "3", str(1 << 40)):                    # every edge a ruler / many / the heads only
            monkeypatch.setenv("MGTA_UT_STRIDE", stride)
            rows, seq = check_unitigs(g, ref)
            if first is None:
                first = rows, seq
            assert np.array_equal(rows, first[0]) and np.array_equal(seq, first[1])
    flags = rows[:, 5]
    if shape == "long":
        assert rows[:, 2].max() > 100_000
    else:
        assert (flags & U.CYCLE).any()


@pytest.mark.gpu
def test_gpu_destinations_repeat_calls_and_queries_afterwards(read_lib):
    import torch
    from megagta_b200 import cabi
    _, rd = read_lib("adversarial")
    k, m = 31, 2
    ref = restated(rd, "adversarial", k, m, 1)
    with build(cabi, rd, k, m, 1, "device") as g:
        rows, seq = check_unitigs(g, ref)
        drows, dseq = g.unitigs(device=True)
        assert drows.is_cuda and dseq.is_cuda and drows.device.index == g.device
        assert np.array_equal(drows.cpu().numpy(), rows) and np.array_equal(dseq.cpu().numpy(), seq)
        r2, s2 = g.unitigs()                                       # twice: the same
        assert np.array_equal(r2, rows) and np.array_equal(s2, seq)
        # straight through the C ABI: device rows with host sequence, and the reverse
        rd_t = torch.empty(rows.size, dtype=torch.int64, device="cuda")
        sh = np.empty_like(seq)
        torch.cuda.synchronize()
        assert g.lib.mgta_sdbg_unitig_copy(g.h, rd_t.data_ptr(), rows.nbytes, sh.ctypes.data, sh.nbytes) == 0
        assert np.array_equal(rd_t.cpu().numpy().reshape(rows.shape), rows) and np.array_equal(sh, seq)
        rh = np.empty_like(rows)
        sd = torch.empty(len(seq), dtype=torch.uint8, device="cuda")
        assert g.lib.mgta_sdbg_unitig_copy(g.h, rh.ctypes.data, rh.nbytes, sd.data_ptr(), len(seq)) == 0
        assert np.array_equal(rh, rows) and np.array_equal(sd.cpu().numpy(), seq)
        edges = np.arange(ref.size, dtype=np.int64)                # the queries still answer after the unitigs
        for op in (R.SQ_FORWARD, R.SQ_REVCOMP, R.SQ_INDEGREE):
            assert np.array_equal(g.query(op, edges), ref.run(op, edges))


@pytest.mark.gpu
def test_gpu_error_paths_leave_the_graph_usable(read_lib):
    import ctypes
    from megagta_b200 import cabi
    _, rd = read_lib("tiny")
    k, m = 25, 2
    ref = restated(rd, "tiny", k, m, 1)
    with cabi.Sdbg(k, True) as g:                                  # before finish
        with pytest.raises(cabi.MgtaError, match="finish"):
            g.unitigs()
    with build(cabi, rd, k, m, 1, "device") as g:
        lib = g.lib
        assert lib.mgta_sdbg_unitig_copy(g.h, None, 0, None, 0) == -4     # copy before compute
        assert b"mgta_sdbg_unitigs first" in lib.mgta_sdbg_last_error(g.h)
        n_rows, n_chars = ctypes.c_int64(), ctypes.c_uint64()
        assert lib.mgta_sdbg_unitigs(g.h, ctypes.byref(n_rows), ctypes.byref(n_chars)) == 0
        rows = np.empty((n_rows.value, 6), np.int64)
        seq = np.empty(n_chars.value, np.uint8)
        assert lib.mgta_sdbg_unitig_copy(g.h, rows.ctypes.data, rows.nbytes - 8, seq.ctypes.data, seq.nbytes) == -1
        assert b"rows buffer" in lib.mgta_sdbg_last_error(g.h)
        assert lib.mgta_sdbg_unitig_copy(g.h, rows.ctypes.data, rows.nbytes, seq.ctypes.data, seq.nbytes - 1) == -1
        assert b"seq buffer" in lib.mgta_sdbg_last_error(g.h)
        assert lib.mgta_sdbg_unitig_copy(g.h, rows.ctypes.data, rows.nbytes, seq.ctypes.data, seq.nbytes) == 0
        want_rows, want_seq = U.restated_unitigs(ref)
        assert np.array_equal(rows, want_rows) and np.array_equal(seq, want_seq)
        check_unitigs(g, ref)
        assert np.array_equal(g.forward(np.arange(ref.size, dtype=np.int64)), ref.fwd)


@pytest.mark.gpu
def test_gpu_fasta_round_trip(read_lib, tmp_path):
    from megagta_b200 import cabi
    _, rd = read_lib("tiny")
    with build(cabi, rd, 25, 2, 1, "device") as g:
        rows, seq = g.unitigs()
    p = str(tmp_path / "unitigs.fa")
    cabi.write_unitigs_fasta(p, rows, seq)
    lines = open(p).read().splitlines()
    assert lines[1::2] == cabi.unitig_strings(rows, seq)
    assert lines[0] == ">unitig_0 len=%d edges=%d multi=%.2f flags=%d" % (25 + rows[0, 2], rows[0, 2], rows[0, 4] / rows[0, 2], rows[0, 5])


@pytest.mark.gpu
def test_gpu_unitig_timing_script_runs():
    script = os.path.join(os.path.dirname(os.path.abspath(__file__)), "gpu_sdbg_unitig_time.py")
    r = subprocess.run(["python3", script, "20000", "31"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["unitigs"] > 0 and line["median_s"] > 0 and line["kernel_share"]
