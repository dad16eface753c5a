"""The device SdBG index (sdbg_index.cu), its navigation queries (sdbg_query.cu, sdbg_nav.cuh) and its unitigs
(sdbg_unitig.cu) against the plain CPU references, on every k and graph the CPU checkers cover: the 52 fuzz inputs of
test_oracle_fuzz.py (k = 9 ... 127 around every word boundary, ragged reads, mercy, assist reads), the random-read matrix
of test_sdbg_query_cpu.py over both build routes and multiplicity modes, graphs of about 10^5 edges at k = 64 and 127,
mercy and assist reads on `tiny`, multiplicities at the 65535 cap, exact palindromes, the hard unitig shapes at
k = 16, 64 and 127 and every ruler stride, and the unitigs of meta200k.

Every graph is compared exactly:
  (a) the index: every section of the device build equals oracle/sdbg_oracle.py's build of the oracle's records;
  (b) every query op on every edge, and LOOKUP on every node label, its reverse complement and seeded absent k-mers,
      equal the numpy restatement (tests/sdbg_query_ref.py);
  (c) the unitig rows and bytes equal the restated rows (tests/sdbg_unitig_ref.py), and the device rows, put in canonical
      form, equal the unitigs compacted straight from the (k+1)-mers of the reads.
test_sdbg_query_cpu.py and test_sdbg_unitig_cpu.py pin the restatements against brute force on the same inputs."""
from collections import Counter

import numpy as np
import pytest

import datasets
import sdbg_query_ref as R
import sdbg_unitig_ref as U
from oracle import oracle as O
from oracle import sdbg_oracle as SO
from test_gpu_sdbg_query import check_all_ops, restated
from test_gpu_sdbg_unitig import check_unitigs
from test_sdbg_index import device_sections
from test_sdbg_query_cpu import RANDOM_KM, fuzz_case, matrix_reads, random_reads

pytestmark = pytest.mark.gpu

CUTS = [0, 1, 3, 777, 16385, 40001, 65535, 65536]                 # host deliveries, cut at odd bucket boundaries
STRIDES = ("1", "3", str(1 << 40))                                 # every edge a ruler / many / the heads only
_REF = {}


class Graph:
    """a read set and what the CPU references make of it"""

    def __init__(self, rd, k, m, need_mercy=False, n_short=None, res=None):
        self.rd, self.k, self.m, self.need_mercy, self.n_short = rd, k, m, need_mercy, n_short
        self.res = res if res is not None else O.build_graph(rd, k, m, need_mercy=need_mercy, n_short=n_short)
        self._sec, self._ref, self._brute = {}, {}, None

    def sections(self, need_mult):
        if need_mult not in self._sec:
            self._sec[need_mult] = SO.build(self.res["stream"], np.asarray(self.res["meta"]), self.k, bool(need_mult))
        return self._sec[need_mult]

    def ref(self, need_mult):
        if need_mult not in self._ref:
            self._ref[need_mult] = R.Restated(self.sections(need_mult), self.k)
        return self._ref[need_mult]

    def brute(self, with_mult):
        """the unitigs compacted from the (k+1)-mers of the reads (U.brute_unitigs), mult_sum None without multiplicities"""
        if self._brute is None:
            self._brute = U.brute_unitigs(R.brute_graph(self.rd, self.k, self.m, self.res["is_solid"], self.n_short), self.k)
        if with_mult:
            return self._brute
        out = Counter()
        for key, n in self._brute.items():
            out[key[:3] + (None,)] += n
        return out

    def build(self, cabi, need_mult, how="device"):
        return build(cabi, self.rd, self.k, self.m, need_mult, how, self.need_mercy, self.n_short)


def build(cabi, rd, k, m, need_mult, how="device", need_mercy=False, n_short=None):
    """the device graph of the reads: stage 1 (m > 1, with mercy edges when asked), stage 2 and the index, the records
    parsed where they lie in HBM (`device`) or handed over from the host in deliveries cut at CUTS (`host`)"""
    g = cabi.Sdbg(k, bool(need_mult))
    try:
        with cabi.Context(k, m, need_mercy=need_mercy, device=0) as ctx:
            ctx.set_reads(rd["seq"], rd["start"], n_short=n_short, max_len=rd["max_len"])
            if m > 1:
                ctx.stage1()
            if how == "device":
                g.from_stage2(ctx)
            else:
                stream, meta, _ = ctx.stage2()
                byts = meta[:, 0] * 2 + meta[:, 2] * 2 + meta[:, 1] * 4 * ((2 * k + 31) // 32)
                off = np.concatenate([[0], np.cumsum(byts)])
                for a, b in zip(CUTS[:-1], CUTS[1:]):
                    g.append(a, b, stream[int(off[a]):int(off[b])], meta[a:b])
        g.finish()
    except BaseException:
        g.close()
        raise
    return g


def cached(key, make):
    if key not in _REF:
        _REF[key] = make()
    return _REF[key]


def check_index_and_queries(g, cabi, gr, need_mult, seed=0):
    """(a) and (b)"""
    got, want = SO.digest(device_sections(g, cabi, need_mult)), SO.digest(gr.sections(need_mult))
    assert set(got) == set(want)
    bad = [s for s in want if got[s] != want[s]]
    assert not bad, bad
    check_all_ops(g, gr.ref(need_mult), need_mult, seed)


def check_rows(g, gr, need_mult):
    """(c) -> the device rows and sequence"""
    rows, seq = check_unitigs(g, gr.ref(need_mult))
    assert U.canonical_rows(rows, seq, gr.k, with_mult=bool(need_mult)) == gr.brute(bool(need_mult))
    return rows, seq


def check_graph(cabi, gr, need_mult, how="device", seed=0):
    with gr.build(cabi, need_mult, how) as g:
        assert g.header().size == gr.ref(need_mult).size
        check_index_and_queries(g, cabi, gr, need_mult, seed)
        return check_rows(g, gr, need_mult)


# ---- the fuzz inputs ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def fuzz_graphs(tmp_path_factory):
    """seed -> Graph, or None for an input without a solid edge"""
    d = str(tmp_path_factory.mktemp("fuzz"))
    out = {}
    for seed in range(52):
        rd, k, m, mercy, n_short, res = fuzz_case(seed, d)
        out[seed] = Graph(rd, k, m, mercy, n_short, res) if res is not None else None
    return out


def test_gpu_fuzz_inputs_with_a_graph_are_most(fuzz_graphs):
    graphs = [gr for gr in fuzz_graphs.values() if gr is not None]
    assert len(graphs) >= 40
    mercy = [gr for gr in graphs if gr.res["num_mercy"]]                 # tiny has no mercy edge: these do
    assert len(mercy) >= 10 and any(gr.n_short is not None for gr in mercy)


@pytest.mark.parametrize("seed", range(52))
def test_gpu_fuzz_inputs(fuzz_graphs, seed):
    from megagta_b200 import cabi
    gr = fuzz_graphs[seed]
    if gr is None:
        pytest.skip("no solid edge")
    # seeds s and s + 26 share k: one of them runs with multiplicities, the other without
    need_mult = int((seed + seed // 26) % 2 == 0)
    check_graph(cabi, gr, need_mult, seed=seed)


# ---- the random-read matrix of the CPU checkers --------------------------------------------------------------------------
@pytest.mark.parametrize("k,m", RANDOM_KM)
@pytest.mark.parametrize("need_mult,how", [(1, "device"), (0, "device"), (1, "host"), (0, "host")])
def test_gpu_random_reads(k, m, need_mult, how):
    from megagta_b200 import cabi
    gr = cached(("matrix", k, m), lambda: Graph(matrix_reads(k, m), k, m))
    check_graph(cabi, gr, need_mult, how, seed=k)


@pytest.mark.parametrize("k", [64, 127])
def test_gpu_graphs_of_1e5_edges_at_large_k(k):
    """rank and select cross major intervals (65536 positions) at wpt = 4 and 8"""
    from megagta_b200 import cabi
    rd = random_reads(5 + k, n_reads=3000, read_len=max(150, k + 40), genome=60000, polya=4, repeats=3, palindromes=20)
    gr = Graph(rd, k, 1)
    assert gr.ref(1).size > 65536
    check_graph(cabi, gr, 1, seed=k)


# ---- mercy, assist reads, multiplicities, palindromes -----------------------------------------------------------------
@pytest.mark.parametrize("assist", [False, True])
@pytest.mark.parametrize("need_mult,how", [(1, "device"), (0, "host")])
def test_gpu_mercy_and_assist_reads(read_lib, data_dir, assist, need_mult, how):
    from megagta_b200 import cabi
    _, rd = read_lib("tiny")
    if assist:
        rd2, n_short = O.with_assist(rd, datasets.assist_fasta("tiny", data_dir))
        gr = cached(("tiny", "assist"), lambda: Graph(rd2, 25, 2, need_mercy=True, n_short=n_short))
    else:
        gr = cached(("tiny", "mercy"), lambda: Graph(rd, 25, 3, need_mercy=True))
    check_graph(cabi, gr, need_mult, how)


def test_gpu_multiplicities_above_254_and_at_the_cap():
    from megagta_b200 import cabi
    gr = Graph(random_reads(7, n_reads=50, read_len=200, genome=600, polya=400, repeats=300), 13, 2)
    with gr.build(cabi, 1) as g:
        check_index_and_queries(g, cabi, gr, 1)
        ref = gr.ref(1)
        mult = g.multiplicity(np.flatnonzero(~ref.invalid))
        assert mult.max() == 65535 and ((mult > 254) & (mult < 65535)).any()
        check_rows(g, gr, 1)                                       # mult_sum too equals the restated sums


def test_gpu_palindromic_edges_and_self_reverse_complement_unitigs():
    from megagta_b200 import cabi
    gr = Graph(random_reads(11, n_reads=40, read_len=64, palindromes=40), 31, 1)   # k + 1 = 32: palindromic edges
    with gr.build(cabi, 1) as g:
        check_index_and_queries(g, cabi, gr, 1)
        valid = np.flatnonzero(~gr.ref(1).invalid)
        assert (g.revcomp(valid) == valid).any()
        rows, _ = check_rows(g, gr, 1)
    assert (rows[:, 5] & U.SELF_RC).any()


# ---- unitig shapes -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", ["long", "circular", "tandem"])
@pytest.mark.parametrize("k", [16, 64, 127])
def test_gpu_unitig_shapes_at_large_and_even_k(shape, k, monkeypatch):
    from megagta_b200 import cabi
    gr = Graph(U.shape_reads(shape, k), k, 1)
    with gr.build(cabi, 1) as g:
        check_index_and_queries(g, cabi, gr, 1, seed=k)
        first = None
        for stride in STRIDES:
            monkeypatch.setenv("MGTA_UT_STRIDE", stride)
            rows, seq = check_unitigs(g, gr.ref(1))
            if first is None:
                first = rows, seq
            assert np.array_equal(rows, first[0]) and np.array_equal(seq, first[1])
        monkeypatch.delenv("MGTA_UT_STRIDE")
        rows, _ = check_rows(g, gr, 1)
    flags = rows[:, 5]
    if shape == "long" and k > 16:                                 # at k = 16 the genome's repeated 16-mers split it
        assert rows[:, 2].max() > 100_000
    if shape == "circular":
        cyc = rows[flags & U.CYCLE == U.CYCLE]
        assert len(cyc) == 1 and cyc[0, 2] == 5000
    if shape == "tandem":
        assert (flags == U.CYCLE | U.SELF_RC).sum() == 3               # the cycles of AT, ACGT and CG


def test_gpu_unitigs_of_meta200k_at_the_default_stride_and_every_edge_a_ruler(read_lib, monkeypatch):
    """at stride 1 the jump rounds run over R = E rulers"""
    from megagta_b200 import cabi
    _, rd = read_lib("meta200k")
    ref = restated(rd, "meta200k", 31, 2, 1)
    with build(cabi, rd, 31, 2, 1) as g:
        rows, seq = check_unitigs(g, ref)
        monkeypatch.setenv("MGTA_UT_STRIDE", "1")
        r1, s1 = check_unitigs(g, ref)
    assert np.array_equal(r1, rows) and np.array_equal(s1, seq)
