"""Links of the unitig graph on the device (include/mgta_sdbg_unitig_graph.h, megagta_b200/csrc/sdbg_unitig.cu) against
the links taken from the unitig strings (tests/sdbg_unitig_graph_ref.py `string_links`), exactly, on the graphs of the
unitig and matrix tests: the query tests' datasets over three build routes and both multiplicity modes, the reference's
own files, the fuzz inputs, 10^5-edge graphs at k = 64 and 127, the unitig shapes at k = 16, 64 and 127, a read set with
hairpins and meta200k.  The device rows are first checked against the restated rows (test_gpu_sdbg_unitig.check_unitigs),
so the strings the links are taken from are the restatement's."""
import ctypes
import json
import os
import subprocess

import numpy as np
import pytest

import sdbg_unitig_graph_ref as G
import sdbg_unitig_ref as U
from oracle import oracle as O
from test_gpu_sdbg_matrix import Graph, build, fuzz_graphs  # noqa: F401  (fuzz_graphs: a fixture)
from test_gpu_sdbg_query import CASES, restated
from test_gpu_sdbg_query import build as build_route
from test_gpu_sdbg_unitig import check_unitigs
from test_sdbg_query_cpu import random_reads

pytestmark = pytest.mark.gpu


def check_links(g, ref):
    """-> device rows, sequence and links, the links equal to string_links of the rows"""
    rows, seq = check_unitigs(g, ref)
    links = g.unitig_links()
    want = G.string_links(rows, seq, ref.k)
    assert links.dtype == np.int64 and links.shape == want.shape, (links.shape, want.shape)
    assert np.array_equal(links, want), np.flatnonzero((links != want).any(axis=1))[:10]
    return rows, seq, links


def self_links_of_cycles(rows, links):
    cyc = np.flatnonzero(rows[:, 5] & U.CYCLE)
    return int(((links[:, 0] == links[:, 1]) & np.isin(links[:, 0] // 2, cyc)).sum())


def links_on_self_rc_rows(rows, links):
    return int(np.isin(links // 2, np.flatnonzero(rows[:, 5] == U.SELF_RC)).any(axis=1).sum())


@pytest.mark.parametrize("ds,k,m", CASES)
@pytest.mark.parametrize("need_mult,how", [(1, "device"), (0, "device"), (1, "host")])
def test_gpu_links_equal_the_string_links(read_lib, ds, k, m, need_mult, how):
    from megagta_b200 import cabi
    _, rd = read_lib(ds)
    with build_route(cabi, rd, k, m, need_mult, how) as g:
        check_links(g, restated(rd, ds, k, m, need_mult))


def test_gpu_links_on_the_files_of_the_reference_buildgraph(read_lib, tmp_path):
    from megagta_b200 import cabi
    if not O.have_ref():
        pytest.skip("oracle/_ref/megagta_ref not built")
    prefix, rd = read_lib("smoke")
    O.run_ref_buildgraph(prefix, str(tmp_path / "ref"), 31, 2)
    with build_route(cabi, rd, 31, 2, 1, "files", tmp_path) as g:
        check_links(g, restated(rd, "smoke", 31, 2, 1))


@pytest.mark.parametrize("seed", range(52))
def test_gpu_links_on_fuzz_inputs(fuzz_graphs, seed):  # noqa: F811
    from megagta_b200 import cabi
    gr = fuzz_graphs[seed]
    if gr is None:
        pytest.skip("no solid edge")
    need_mult = int((seed + seed // 26) % 2 == 0)
    with gr.build(cabi, need_mult) as g:
        check_links(g, gr.ref(need_mult))


@pytest.mark.parametrize("k", [64, 127])
def test_gpu_links_on_graphs_of_1e5_edges_at_large_k(k):
    from megagta_b200 import cabi
    gr = Graph(random_reads(5 + k, n_reads=3000, read_len=max(150, k + 40), genome=60000, polya=4, repeats=3, palindromes=20), k, 1)
    assert gr.ref(1).size > 65536
    with gr.build(cabi, 1) as g:
        _, _, links = check_links(g, gr.ref(1))
    assert len(links)


@pytest.mark.parametrize("shape", ["long", "circular", "tandem"])
@pytest.mark.parametrize("k", [16, 64, 127])
def test_gpu_links_on_the_unitig_shapes(shape, k):
    from megagta_b200 import cabi
    gr = Graph(U.shape_reads(shape, k), k, 1)
    with gr.build(cabi, 1) as g:
        rows, _, links = check_links(g, gr.ref(1))
    if shape != "long":
        assert self_links_of_cycles(rows, links) == int((rows[:, 5] & U.CYCLE).astype(bool).sum()) > 0
    if shape == "tandem":
        assert (links[:, 0] == links[:, 1])[np.isin(links[:, 0] // 2, np.flatnonzero(rows[:, 5] == U.CYCLE | U.SELF_RC))].sum() == 3


@pytest.mark.parametrize("need_mult,how", [(1, "device"), (0, "host")])
def test_gpu_hairpins_and_links_of_self_reverse_complement_rows(need_mult, how):
    """a -> bar(a) needs a palindromic node, so an even k"""
    from megagta_b200 import cabi
    gr = Graph(G.hairpin_reads(), 16, 1)
    with gr.build(cabi, need_mult, how) as g:
        rows, _, links = check_links(g, gr.ref(need_mult))
    assert len(G.hairpins(rows, links)) >= 2 and links_on_self_rc_rows(rows, links) >= 2


def test_gpu_links_of_meta200k(read_lib):
    from megagta_b200 import cabi
    _, rd = read_lib("meta200k")
    with build(cabi, rd, 31, 2, 1) as g:
        rows, _, links = check_links(g, restated(rd, "meta200k", 31, 2, 1))
    assert len(links) > 1000 and (links[:, 0] & 1).any() and (links[:, 1] & 1).any()


def test_gpu_destinations_repeat_calls_and_links_after_new_unitigs(read_lib, monkeypatch):
    import torch
    from megagta_b200 import cabi
    _, rd = read_lib("adversarial")
    ref = restated(rd, "adversarial", 31, 2, 1)
    with build(cabi, rd, 31, 2, 1) as g:
        rows, seq, links = check_links(g, ref)
        d = g.unitig_links(device=True)
        assert d.is_cuda and d.device.index == g.device and d.dtype == torch.int64
        assert np.array_equal(d.cpu().numpy(), links)
        assert np.array_equal(g.unitig_links(), links)               # twice: the same
        raw = torch.empty(links.size, dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()
        assert g.lib.mgta_sdbg_unitig_link_copy(g.h, raw.data_ptr(), links.nbytes) == 0    # copy again, no new compute
        assert np.array_equal(raw.cpu().numpy().reshape(links.shape), links)
        monkeypatch.setenv("MGTA_UT_STRIDE", "1")                  # new unitigs (the same rows), then their links
        r2, s2, l2 = check_links(g, ref)
        assert np.array_equal(r2, rows) and np.array_equal(s2, seq) and np.array_equal(l2, links)
        rh, sh = np.empty_like(rows), np.empty_like(seq)           # the links leave the rows and bytes as they were
        assert g.lib.mgta_sdbg_unitig_copy(g.h, rh.ctypes.data, rh.nbytes, sh.ctypes.data, sh.nbytes) == 0
        assert np.array_equal(rh, rows) and np.array_equal(sh, seq)


def test_gpu_error_paths_leave_the_graph_usable(read_lib):
    from megagta_b200 import cabi
    _, rd = read_lib("adversarial")
    ref = restated(rd, "adversarial", 31, 2, 1)
    n = ctypes.c_int64()
    with cabi.Sdbg(31, True) as g:                                  # before finish
        assert g.lib.mgta_sdbg_unitig_links(g.h, ctypes.byref(n)) == -4
        with pytest.raises(cabi.MgtaError, match="mgta_sdbg_unitigs first"):
            g.unitig_links()
    with build(cabi, rd, 31, 2, 1) as g:
        lib = g.lib
        assert lib.mgta_sdbg_unitig_links(g.h, ctypes.byref(n)) == -4      # before the unitigs
        assert b"mgta_sdbg_unitigs first" in lib.mgta_sdbg_last_error(g.h)
        assert lib.mgta_sdbg_unitig_link_copy(g.h, None, 0) == -4
        rows, seq = g.unitigs()
        assert lib.mgta_sdbg_unitig_link_copy(g.h, None, 0) == -4           # unitigs, but no links yet
        assert b"mgta_sdbg_unitig_links" in lib.mgta_sdbg_last_error(g.h)
        assert lib.mgta_sdbg_unitig_links(g.h, None) == -1
        assert b"null n_links" in lib.mgta_sdbg_last_error(g.h)
        assert lib.mgta_sdbg_unitig_links(g.h, ctypes.byref(n)) == 0
        links = np.empty((n.value, 2), np.int64)
        assert len(links)
        assert lib.mgta_sdbg_unitig_link_copy(g.h, links.ctypes.data, links.nbytes - 8) == -1
        assert b"links buffer of %d bytes, %d needed" % (links.nbytes - 8, links.nbytes) in lib.mgta_sdbg_last_error(g.h)
        assert lib.mgta_sdbg_unitig_link_copy(g.h, None, links.nbytes) == -1
        assert lib.mgta_sdbg_unitig_link_copy(g.h, links.ctypes.data, links.nbytes) == 0
        assert np.array_equal(links, G.string_links(rows, seq, 31))
        g.unitigs()                                                # new rows: the old links are stale
        assert lib.mgta_sdbg_unitig_link_copy(g.h, links.ctypes.data, links.nbytes) == -4
        check_links(g, ref)
        assert np.array_equal(g.forward(np.arange(ref.size, dtype=np.int64)), ref.fwd)


def test_gpu_gfa_round_trip(read_lib, tmp_path):
    from megagta_b200 import cabi
    _, rd = read_lib("adversarial")
    k = 31
    with build(cabi, rd, k, 2, 1) as g:
        rows, seq = g.unitigs()
        links = g.unitig_links()
    p = str(tmp_path / "unitigs.gfa")
    cabi.write_unitigs_gfa(p, rows, seq, links, k)
    lines = open(p).read().splitlines()
    assert lines[0] == "H\tVN:Z:1.0"
    S = [ln.split("\t") for ln in lines if ln[0] == "S"]
    L = [ln.split("\t") for ln in lines if ln[0] == "L"]
    strings = cabi.unitig_strings(rows, seq)
    assert [s[2] for s in S] == strings and [s[1] for s in S] == ["unitig_%d" % r for r in range(len(rows))]
    assert all(s[3] == "LN:i:%d" % len(s[2]) and s[4] == "KC:i:%d" % rows[r, 4] for r, s in enumerate(S))
    assert len(L) == len(links) > 0
    by_name = {s[1]: s[2] for s in S}

    def oriented(name, o):
        s = by_name[name]
        return s if o == "+" else s[::-1].translate(str.maketrans("ACGT", "TGCA"))

    for _, a, oa, b, ob, ov in L:
        assert ov == "%dM" % k
        assert oriented(a, oa)[-k:] == oriented(b, ob)[:k]


def test_gpu_unitig_graph_timing_script_runs():
    script = os.path.join(os.path.dirname(os.path.abspath(__file__)), "gpu_sdbg_unitig_graph_time.py")
    r = subprocess.run(["python3", script, "20000", "31"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["unitigs"] > 0 and line["links"] >= 0 and line["median_s"] > 0 and line["kernel_share"] and line["same_after_copy"]
