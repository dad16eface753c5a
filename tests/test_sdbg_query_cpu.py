"""Navigation queries on the SdBG (include/mgta_sdbg_query.h) without a GPU.

The numpy restatement of every op (tests/sdbg_query_ref.py `Restated`, over the reference's own arrays as
oracle/sdbg_oracle.py rebuilds them) against the de Bruijn graph taken straight from the reads (`brute_graph`), and the
C ABI of the new header the way test_abi_cpu.py checks include/mgta_cuda.h."""
import ctypes
import os
import re

import numpy as np
import pytest

import datasets
import sdbg_query_ref as R
from oracle import oracle as O
from oracle import sdbg_oracle as SO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def random_reads(seed, n_reads=300, read_len=90, genome=3000, polya=0, repeats=0, palindromes=0):
    """reads of a small random genome (both strands), poly-A reads, `repeats` copies of one read and exact palindromes ->
    the read dict oracle.load_read_lib returns"""
    rng = np.random.default_rng(seed)
    g = rng.integers(0, 4, size=genome, dtype=np.uint8)
    reads = []
    for p in rng.integers(0, genome - read_len, size=n_reads):
        r = g[p:p + read_len]
        reads.append(r if rng.integers(2) else (3 - r)[::-1])
    reads += [np.zeros(read_len, np.uint8)] * polya
    reads += [g[:read_len]] * repeats
    for _ in range(palindromes):
        h = rng.integers(0, 4, size=read_len // 2, dtype=np.uint8)
        reads.append(np.concatenate([h, (3 - h)[::-1]]))
    lens = np.array([len(r) for r in reads], np.int64)
    start = np.zeros(len(reads) + 1, np.uint64)
    start[1:] = np.cumsum(lens)
    seq, start = O.pack_reversed(np.concatenate(reads).astype(np.uint8), start)
    return dict(seq=seq, start=start, n_reads=len(reads), max_len=int(lens.max()))


RANDOM_KM = [(13, 1), (15, 2), (16, 3), (17, 2), (31, 1), (32, 2), (33, 3), (63, 2), (64, 1), (127, 2)]


def matrix_reads(k, m):
    """the random read set of the (k, m) cell of RANDOM_KM"""
    return random_reads(1000 + k * 10 + m, read_len=max(90, k + 40), polya=4, repeats=3, palindromes=6)


def fuzz_case(seed, d):
    """the read set of test_oracle_fuzz.make_case(seed) (files under d), its assist reads appended when the case has any
    -> (reads, k, m, need_mercy, n_short, the oracle's build_graph of it or None when it has no solid edge)"""
    import test_oracle_fuzz as F
    prefix, k, m, mercy, fa = F.make_case(seed, d)
    rd, n_short = O.load_read_lib(prefix), None
    if fa:
        rd, n_short = O.with_assist(rd, fa)
    res = O.build_graph(rd, k, m, need_mercy=mercy, n_short=n_short)
    return rd, k, m, mercy, n_short, (res if int(res["meta"][:, 0].sum()) else None)


def check_against_brute_force(rd, k, m, need_mercy=False, n_short=None, absent=2000, seed=0):
    res = O.build_graph(rd, k, m, need_mercy=need_mercy, n_short=n_short)
    ref = R.Restated(SO.build(res["stream"], np.asarray(res["meta"]), k, True), k)
    E = R.brute_graph(rd, k, m, res["is_solid"], n_short)
    valid = np.flatnonzero(~ref.invalid)
    assert len(valid) == len(E)
    ek = {ref.edge_kmers[e].tobytes(): int(e) for e in valid}
    assert set(ek) == set(E)
    # multiplicities equal the solid-occurrence counts
    mult = ref.run(R.SQ_MULTIPLICITY, valid)
    assert all(E[ref.edge_kmers[e].tobytes()] == mult[j] for j, e in enumerate(valid))
    # LOOKUP finds exactly the prefixes and suffixes of the edges; LABEL(LOOKUP(X)) = X
    nodes = sorted({x[:k] for x in E} | {x[1:] for x in E})
    X = np.frombuffer(b"".join(nodes), np.uint8).reshape(-1, k) if nodes else np.zeros((0, k), np.uint8)
    found = ref.run(R.SQ_LOOKUP, R.pack_chars(X))
    assert (found >= 0).all()
    assert ref.last[found].all() and not ref.tip[found].any()
    lab = ref.run(R.SQ_LABEL, found)
    assert np.array_equal(lab[:, :-1], R.pack_chars(X)) and not lab[:, -1].any()
    rng = np.random.default_rng(seed)
    Y = rng.integers(0, 4, size=(absent, k), dtype=np.uint8)
    node_set = set(nodes)
    want = np.array([y.tobytes() in node_set for y in Y])
    assert np.array_equal(ref.run(R.SQ_LOOKUP, R.pack_chars(Y)) >= 0, want)
    # degrees: |{c : X.c in E}| and |{c : c.X in E}|
    od = ref.run(R.SQ_OUTDEGREE, found)
    idg = ref.run(R.SQ_INDEGREE, found)
    for j, x in enumerate(nodes):
        assert od[j] == sum((x + bytes([c])) in E for c in range(4))
        assert idg[j] == sum((bytes([c]) + x) in E for c in range(4))
    out = ref.run(R.SQ_OUTGOING, found)
    inc = ref.run(R.SQ_INCOMING, found)
    assert np.array_equal((out >= 0).sum(axis=1), od) and np.array_equal((inc >= 0).sum(axis=1), idg)
    assert all(ref.edge_kmers[e][:k].tobytes() == nodes[j] for j in range(len(nodes)) for e in out[j] if e >= 0)
    assert all(ref.edge_kmers[e][1:].tobytes() == nodes[j] for j in range(len(nodes)) for e in inc[j] if e >= 0)
    # LABEL(FORWARD(i)) = LABEL(i)[1:] + W(i), BACKWARD leads into v(i)
    fw = ref.run(R.SQ_FORWARD, valid)
    assert np.array_equal(ref.lab[fw], ref.edge_kmers[valid][:, 1:])
    real = np.flatnonzero(~ref.tip)
    bw = ref.run(R.SQ_BACKWARD, real)
    assert np.array_equal(ref.fwd[bw], ref.last_pos[ref.node[real]])
    assert (ref.W[bw] >= 1).all() and (ref.W[bw] <= 4).all()
    # REVCOMP: an involution on valid edges that matches the reverse complement of the (k+1)-mer
    rc = ref.run(R.SQ_REVCOMP, valid)
    assert (rc >= 0).all()
    assert np.array_equal(ref.run(R.SQ_REVCOMP, rc), valid)
    assert np.array_equal(ref.edge_kmers[rc], (3 - ref.edge_kmers[valid])[:, ::-1])
    assert (ref.run(R.SQ_REVCOMP, np.flatnonzero(ref.invalid)) == -1).all()
    # tip nodes: '$' + k - 1 characters, no valid edges
    tips = np.flatnonzero(ref.tip)
    assert (ref.run(R.SQ_LABEL, tips)[:, -1] == 1).all()
    assert (ref.run(R.SQ_OUTDEGREE, tips) == 0).all() and (ref.run(R.SQ_BACKWARD, tips) == -1).all()
    return ref


@pytest.mark.parametrize("ds,k,m", [("tiny", 25, 2), ("smoke", 13, 2), ("adversarial", 31, 2), ("adversarial", 16, 1),
                                    ("xander", 29, 1)])
def test_restatement_equals_brute_force_on_datasets(read_lib, ds, k, m):
    _, rd = read_lib(ds)
    if ds == "smoke":                                              # 2000 of the 20 k reads: the python checks stay quick
        n = 2000
        rd = dict(rd, n_reads=n, start=rd["start"][:n + 1].copy())
    check_against_brute_force(rd, k, m)


@pytest.mark.parametrize("k,m", RANDOM_KM)
def test_restatement_equals_brute_force_on_random_reads(k, m):
    check_against_brute_force(matrix_reads(k, m), k, m, seed=k)


@pytest.mark.parametrize("seed", range(52))
def test_restatement_equals_brute_force_on_fuzz_inputs(seed, tmp_path):
    """k = 9 ... 127 around every word boundary, ragged reads, errors, mercy and assist reads"""
    rd, k, m, mercy, n_short, res = fuzz_case(seed, str(tmp_path))
    if res is None:
        pytest.skip("no solid edge")
    check_against_brute_force(rd, k, m, need_mercy=mercy, n_short=n_short, absent=300, seed=seed)


def test_most_fuzz_inputs_have_a_graph(tmp_path):
    assert sum(fuzz_case(seed, str(tmp_path))[-1] is not None for seed in range(52)) >= 40


def test_mercy_and_assist_reads(read_lib, data_dir):
    _, rd = read_lib("tiny")
    check_against_brute_force(rd, 25, 3, need_mercy=True)
    rd2, n_short = O.with_assist(rd, datasets.assist_fasta("tiny", data_dir))
    check_against_brute_force(rd2, 25, 2, need_mercy=True, n_short=n_short)


def test_multiplicities_above_254_and_at_the_cap():
    rd = random_reads(7, n_reads=50, read_len=200, genome=600, polya=400, repeats=300)
    ref = check_against_brute_force(rd, 13, 2)
    assert ref.mult.max() == 65535 and ((ref.mult > 254) & (ref.mult < 65535)).any()


def test_palindromic_edges_are_their_own_reverse_complement():
    rd = random_reads(11, n_reads=40, read_len=64, palindromes=40)
    ref = check_against_brute_force(rd, 31, 1)                   # k + 1 = 32: even (k+1)-mers can be palindromes
    valid = np.flatnonzero(~ref.invalid)
    assert (ref.run(R.SQ_REVCOMP, valid) == valid).any()


# ---- the C ABI of include/mgta_sdbg_query.h ------------------------------------------------------------------------
def declared():
    txt = open(os.path.join(ROOT, "include", "mgta_sdbg_query.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(mgta_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_query_entry_point():
    from megagta_b200 import cabi
    lib = ctypes.CDLL(cabi.LIB_PATH)
    names = declared()
    assert names == ["mgta_sdbg_query", "mgta_sdbg_query_row_bytes"]
    assert not [n for n in names if not hasattr(lib, n)]


def test_query_binding_covers_the_header_and_declares_argtypes():
    from megagta_b200 import cabi
    assert sorted(cabi.QUERY_EXPORTS) == declared()
    assert not set(cabi.QUERY_EXPORTS) & set(cabi.EXPORTS)
    lib = cabi.load()
    assert all(getattr(lib, n).argtypes is not None for n in cabi.QUERY_EXPORTS)
    txt = open(os.path.join(ROOT, "include", "mgta_sdbg_query.h")).read()
    ops = re.findall(r"\b(MGTA_SQ_[A-Z]+)\b", txt)
    names = list(dict.fromkeys(ops))
    assert [getattr(cabi, n[5:]) for n in names] == list(range(1, 11))
    assert cabi.SQ_LOOKUP == R.SQ_LOOKUP and cabi.SQ_REVCOMP == R.SQ_REVCOMP


def test_no_device_means_an_error_not_a_fallback():
    import torch
    from megagta_b200 import cabi
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    lib = cabi.load()
    a, b = ctypes.c_uint64(), ctypes.c_uint64()
    assert lib.mgta_sdbg_query_row_bytes(None, cabi.SQ_LOOKUP, ctypes.byref(a), ctypes.byref(b)) == -1
    assert lib.mgta_sdbg_query(None, cabi.SQ_FORWARD, None, 0, None, 0) == -1
    with pytest.raises(cabi.MgtaError):                            # no graph, hence no query, without a device
        cabi.Sdbg(31)


def test_kmer_string_helpers():
    from megagta_b200 import cabi
    rng = np.random.default_rng(5)
    for k in (13, 15, 16, 17, 31, 32, 33, 63, 64, 127):
        s = ["".join("ACGT"[c] for c in rng.integers(0, 4, size=k)) for _ in range(20)]
        p = cabi.pack_kmers(s, k)
        assert p.shape == (20, (2 * k + 31) // 32) and cabi.unpack_kmers(p, k) == s
        assert np.array_equal(p, R.pack_chars(np.array([[("ACGT".index(c)) for c in x] for x in s], np.uint8)))
    assert cabi.pack_kmers(["C" + "A" * 12], 13)[0, 0] == 1 << 30
    with pytest.raises(ValueError):
        cabi.pack_kmers(["ACGN" + "A" * 9], 13)
