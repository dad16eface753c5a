"""Unitigs of the SdBG (include/mgta_sdbg_unitig.h) without a GPU.

The restated rows (tests/sdbg_unitig_ref.py `restated_unitigs`, over the numpy restatement of the navigation queries)
against the unitigs compacted straight from the k-mer strings of the reads (`brute_unitigs`), on the matrix of
test_sdbg_query_cpu.py and on read sets with a very long unitig, a long cycle and short cycles; and the C ABI of the new
header the way test_sdbg_query_cpu.py checks its own."""
import ctypes
import os
import re

import numpy as np
import pytest

import datasets
import sdbg_query_ref as R
import sdbg_unitig_ref as U
from oracle import oracle as O
from oracle import sdbg_oracle as SO
from test_sdbg_query_cpu import random_reads

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def check_against_brute_force(rd, k, m, need_mercy=False, n_short=None):
    res = O.build_graph(rd, k, m, need_mercy=need_mercy, n_short=n_short)
    ref = R.Restated(SO.build(res["stream"], np.asarray(res["meta"]), k, True), k)
    rows, seq = U.restated_unitigs(ref)
    n_valid = int((~ref.invalid).sum())
    assert U.edge_invariant(rows) == n_valid
    assert (np.diff(rows[:, 0]) > 0).all()
    assert rows[:, 3].tolist() == np.concatenate([[0], np.cumsum(k + rows[:, 2])[:-1]]).tolist() and len(seq) == (k + rows[:, 2]).sum()
    assert U.canonical_rows(rows, seq, k) == U.brute_unitigs(R.brute_graph(rd, k, m, res["is_solid"], n_short), k)
    cyc = rows[rows[:, 5] & U.CYCLE == U.CYCLE]
    for r in cyc:                                                  # a cycle's last k characters repeat its first k
        s = seq[r[3]:r[3] + k + r[2]]
        assert np.array_equal(s[:k], s[-k:])
    return ref, rows, seq


@pytest.mark.parametrize("ds,k,m", [("tiny", 25, 2), ("smoke", 13, 2), ("adversarial", 31, 2), ("adversarial", 16, 1),
                                    ("xander", 29, 1)])
def test_restated_unitigs_equal_brute_force_on_datasets(read_lib, ds, k, m):
    _, rd = read_lib(ds)
    if ds == "smoke":
        n = 2000
        rd = dict(rd, n_reads=n, start=rd["start"][:n + 1].copy())
    check_against_brute_force(rd, k, m)


@pytest.mark.parametrize("k,m", [(13, 1), (15, 2), (16, 3), (17, 2), (31, 1), (32, 2), (33, 3), (63, 2), (64, 1), (127, 2)])
def test_restated_unitigs_equal_brute_force_on_random_reads(k, m):
    rd = random_reads(1000 + k * 10 + m, read_len=max(90, k + 40), polya=4, repeats=3, palindromes=6)
    check_against_brute_force(rd, k, m)


def test_mercy_and_assist_reads(read_lib, data_dir):
    _, rd = read_lib("tiny")
    check_against_brute_force(rd, 25, 3, need_mercy=True)
    rd2, n_short = O.with_assist(rd, datasets.assist_fasta("tiny", data_dir))
    check_against_brute_force(rd2, 25, 2, need_mercy=True, n_short=n_short)


def test_palindromes_give_self_reverse_complement_unitigs():
    rd = random_reads(11, n_reads=40, read_len=64, palindromes=40)
    _, rows, _ = check_against_brute_force(rd, 31, 1)
    assert (rows[:, 5] & U.SELF_RC).any()


def test_one_long_genome_is_one_unitig_pair():
    rd = U.long_genome_reads()
    _, rows, _ = check_against_brute_force(rd, 31, 1)
    assert rows[:, 2].max() > 100_000


def test_circular_genome_is_a_cycle_longer_than_any_stride():
    _, rows, _ = check_against_brute_force(U.circular_genome_reads(), 31, 1)
    cyc = rows[rows[:, 5] & U.CYCLE == U.CYCLE]
    assert len(cyc) == 1 and cyc[0, 2] == 5000


def test_tandem_repeats_give_short_cycles():
    _, rows, _ = check_against_brute_force(U.tandem_reads(), 21, 1)
    cyc = rows[rows[:, 5] & U.CYCLE == U.CYCLE]
    assert sorted(cyc[:, 2].tolist()) == [1, 2, 5, 7, 13]            # poly-A is a self-loop (and poly-T its partner)


# ---- the C ABI of include/mgta_sdbg_unitig.h -----------------------------------------------------------------------
def declared():
    txt = open(os.path.join(ROOT, "include", "mgta_sdbg_unitig.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(mgta_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_unitig_entry_point():
    from megagta_b200 import cabi
    lib = ctypes.CDLL(cabi.LIB_PATH)
    names = declared()
    assert names == ["mgta_sdbg_unitig_copy", "mgta_sdbg_unitigs"]
    assert not [n for n in names if not hasattr(lib, n)]


def test_unitig_binding_covers_the_header_and_declares_argtypes():
    from megagta_b200 import cabi
    assert sorted(cabi.UNITIG_EXPORTS) == declared()
    assert not set(cabi.UNITIG_EXPORTS) & (set(cabi.EXPORTS) | set(cabi.QUERY_EXPORTS))
    lib = cabi.load()
    assert all(getattr(lib, n).argtypes is not None for n in cabi.UNITIG_EXPORTS)
    assert (cabi.UNITIG_CYCLE, cabi.UNITIG_SELF_RC) == (U.CYCLE, U.SELF_RC)


def test_no_device_means_an_error_not_a_fallback():
    import torch
    from megagta_b200 import cabi
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    lib = cabi.load()
    a, b = ctypes.c_int64(), ctypes.c_uint64()
    assert lib.mgta_sdbg_unitigs(None, ctypes.byref(a), ctypes.byref(b)) == -1
    assert lib.mgta_sdbg_unitig_copy(None, None, 0, None, 0) == -1


def test_fasta_writer_and_strings(tmp_path):
    from megagta_b200 import cabi
    seq = np.frombuffer(b"ACGTACGTTTTTGGGA", np.uint8)
    rows = np.array([[0, 3, 4, 0, 10, 0], [5, 5, 1, 8, -1, 2], [9, 9, 4, 13, 8, 1]], np.int64)
    assert cabi.unitig_strings(rows, seq) == ["ACGTACGT", "TTTTG", "GGA"]
    p = tmp_path / "u.fa"
    cabi.write_unitigs_fasta(str(p), rows, seq, min_len=6)
    assert p.read_text() == ">unitig_0 len=8 edges=4 multi=2.50 flags=0\nACGTACGT\n"
    cabi.write_unitigs_fasta(str(p), rows, seq)
    assert p.read_text().splitlines()[2] == ">unitig_1 len=5 edges=1 multi=na flags=2"
