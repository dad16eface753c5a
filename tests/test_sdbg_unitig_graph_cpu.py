"""Links of the unitig graph (include/mgta_sdbg_unitig_graph.h) without a GPU.

The links taken from the unitig strings (tests/sdbg_unitig_graph_ref.py `string_links`, over the restated rows of
tests/sdbg_unitig_ref.py) against a restatement of the header's definition on edges (`edge_links`: ends, FORWARD,
OUTGOING and REVCOMP of the numpy restatement of the queries), on the inputs of test_sdbg_unitig_cpu.py and on a read set
with hairpins; the C ABI of the new header; the GFA writer."""
import ctypes
import os
import re

import numpy as np
import pytest

import datasets
import sdbg_query_ref as R
import sdbg_unitig_graph_ref as G
import sdbg_unitig_ref as U
from oracle import oracle as O
from oracle import sdbg_oracle as SO
from test_sdbg_query_cpu import RANDOM_KM, fuzz_case, matrix_reads, random_reads

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def edge_links(ref, rows):
    """the header's definition on edge ids: id of every head, end of every linear oriented unitig, FORWARD and OUTGOING
    there; (2r, 2r) and its twin per cycle -> the canonical links"""
    lin = np.flatnonzero(rows[:, 5] & U.CYCLE == 0)
    two = lin[rows[lin, 5] & U.SELF_RC == 0]
    hid = np.full(ref.size, -1, np.int64)
    hid[rows[lin, 0]] = 2 * lin
    hid[ref.run(R.SQ_REVCOMP, rows[two, 1])] = 2 * two + 1
    a = np.concatenate([2 * lin, 2 * two + 1])
    end = np.concatenate([rows[lin, 1], ref.run(R.SQ_REVCOMP, rows[two, 0])])
    out = ref.out_tab[ref.node[ref.fwd[end]]]
    assert (hid[out[out >= 0]] >= 0).all()                         # every out-edge there starts a linear unitig
    F = {(int(x), int(hid[f])) for x, fs in zip(a.tolist(), out.tolist()) for f in fs if f >= 0}
    for r in np.flatnonzero(rows[:, 5] & U.CYCLE).tolist():
        F |= {(2 * r, 2 * r), (G.bar(rows, 2 * r), G.bar(rows, 2 * r))}
    return G.canonical_links(rows, F)


def check_links(rd, k, m, need_mercy=False, n_short=None):
    res = O.build_graph(rd, k, m, need_mercy=need_mercy, n_short=n_short)
    ref = R.Restated(SO.build(res["stream"], np.asarray(res["meta"]), k, True), k)
    rows, seq = U.restated_unitigs(ref)
    F = G.all_string_links(rows, seq, k)
    assert all((G.bar(rows, b), G.bar(rows, a)) in F for a, b in F)
    links = G.string_links(rows, seq, k)
    assert np.array_equal(links, edge_links(ref, rows))
    assert len(np.unique(links, axis=0)) == len(links)
    return rows, links


@pytest.mark.parametrize("k,m", RANDOM_KM)
def test_links_on_random_reads(k, m):
    check_links(matrix_reads(k, m), k, m)


@pytest.mark.parametrize("seed", range(52))
def test_links_on_fuzz_inputs(seed, tmp_path):
    rd, k, m, mercy, n_short, res = fuzz_case(seed, str(tmp_path))
    if res is None:
        pytest.skip("no solid edge")
    check_links(rd, k, m, need_mercy=mercy, n_short=n_short)


def test_links_with_mercy_and_assist_reads(read_lib, data_dir):
    _, rd = read_lib("tiny")
    check_links(rd, 25, 3, need_mercy=True)
    rd2, n_short = O.with_assist(rd, datasets.assist_fasta("tiny", data_dir))
    check_links(rd2, 25, 2, need_mercy=True, n_short=n_short)


def test_links_on_palindromes():
    check_links(random_reads(11, n_reads=40, read_len=64, palindromes=40), 31, 1)


@pytest.mark.parametrize("shape", ["long", "circular", "tandem"])
@pytest.mark.parametrize("k", [16, 64, 127])
def test_links_on_the_unitig_shapes(shape, k):
    rows, links = check_links(U.shape_reads(shape, k), k, 1)
    cyc = np.flatnonzero(rows[:, 5] & U.CYCLE)
    if len(cyc):                                                    # every cycle links to itself, and to nothing else
        assert {(2 * r, 2 * r) for r in cyc.tolist()} <= set(map(tuple, links.tolist()))
        assert not np.isin(links // 2, cyc).any(axis=1)[links[:, 0] != links[:, 1]].any()


def test_hairpins_and_links_of_self_reverse_complement_rows():
    rows, links = check_links(G.hairpin_reads(), 16, 1)
    assert G.hairpins(rows, links)
    self_rc = np.flatnonzero(rows[:, 5] == U.SELF_RC)
    assert np.isin(links // 2, self_rc).any()


# ---- the C ABI of include/mgta_sdbg_unitig_graph.h -----------------------------------------------------------------
def declared():
    txt = open(os.path.join(ROOT, "include", "mgta_sdbg_unitig_graph.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(mgta_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_unitig_graph_entry_point():
    from megagta_b200 import cabi
    lib = ctypes.CDLL(cabi.LIB_PATH)
    names = declared()
    assert names == ["mgta_sdbg_unitig_link_copy", "mgta_sdbg_unitig_links"]
    assert not [n for n in names if not hasattr(lib, n)]


def test_unitig_graph_binding_covers_the_header_and_declares_argtypes():
    from megagta_b200 import cabi
    assert sorted(cabi.UNITIG_GRAPH_EXPORTS) == declared()
    assert not set(cabi.UNITIG_GRAPH_EXPORTS) & (set(cabi.EXPORTS) | set(cabi.QUERY_EXPORTS) | set(cabi.UNITIG_EXPORTS))
    lib = cabi.load()
    assert all(getattr(lib, n).argtypes is not None for n in cabi.UNITIG_GRAPH_EXPORTS)


def test_no_device_means_an_error_not_a_fallback():
    import torch
    from megagta_b200 import cabi
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    lib = cabi.load()
    n = ctypes.c_int64()
    assert lib.mgta_sdbg_unitig_links(None, ctypes.byref(n)) == -1
    assert lib.mgta_sdbg_unitig_link_copy(None, None, 0) == -1


def test_gfa_writer(tmp_path):
    from megagta_b200 import cabi
    seq = np.frombuffer(b"ACGTACGTTTTTGGGA", np.uint8)
    rows = np.array([[0, 3, 4, 0, 10, 0], [5, 5, 1, 8, -1, 2], [9, 9, 4, 13, 8, 1]], np.int64)
    links = np.array([[0, 2], [1, 4], [4, 4]], np.int64)
    p = tmp_path / "u.gfa"
    cabi.write_unitigs_gfa(str(p), rows, seq, links, 2)
    assert p.read_text() == ("H\tVN:Z:1.0\n"
                             "S\tunitig_0\tACGTACGT\tLN:i:8\tKC:i:10\n"
                             "S\tunitig_1\tTTTTG\tLN:i:5\n"
                             "S\tunitig_2\tGGA\tLN:i:3\tKC:i:8\n"
                             "L\tunitig_0\t+\tunitig_1\t+\t2M\n"
                             "L\tunitig_0\t-\tunitig_2\t+\t2M\n"
                             "L\tunitig_2\t+\tunitig_2\t+\t2M\n")


def test_string_links_on_hand_made_rows():
    # k = 3; oriented: 0 AACGT, 1 ACGTT, 2 CGTT, 3 AACG, and the self-reverse-complement cycle 4 ACGTAC.  F holds
    # (0, 2) and its twin (3, 1), and (4, 4)
    seq = np.frombuffer(b"AACGTCGTTACGTAC", np.uint8)
    rows = np.array([[0, 1, 2, 0, -1, 0], [2, 2, 1, 5, -1, 0], [3, 3, 3, 9, -1, 3]], np.int64)
    assert G.all_string_links(rows, seq, 3) == {(0, 2), (3, 1), (4, 4)}
    assert G.string_links(rows, seq, 3).tolist() == [[0, 2], [4, 4]]
