"""TEST INFRASTRUCTURE ONLY: two checkers for the navigation queries of include/mgta_sdbg_query.h.

- `Restated`: a vectorised numpy restatement of every op over the sections that oracle/sdbg_oracle.py `build()` returns
  (the reference's own arrays).  It works through whole-array prefix sums and the forward map instead of per-row rank /
  select chains, so it shares no logic with the kernels (megagta_b200/csrc/sdbg_query.cu).
- `brute_graph`: the de Bruijn graph straight from the reads and `is_solid`, closed under reverse complement.
"""
import numpy as np

from oracle import oracle as O

SQ_LOOKUP, SQ_LABEL, SQ_FORWARD, SQ_BACKWARD, SQ_OUTDEGREE, SQ_INDEGREE, SQ_OUTGOING, SQ_INCOMING, SQ_MULTIPLICITY, SQ_REVCOMP = range(1, 11)
EDGE_OPS = [SQ_LABEL, SQ_FORWARD, SQ_BACKWARD, SQ_OUTDEGREE, SQ_INDEGREE, SQ_OUTGOING, SQ_INCOMING, SQ_MULTIPLICITY, SQ_REVCOMP]
ACGT = np.frombuffer(b"ACGT", np.uint8)


def _bits(b, n):
    return np.unpackbits(np.frombuffer(b, np.uint8), bitorder="little")[:n].astype(bool)


def pack_chars(c):
    """uint8 [n, k] characters 0..3 -> uint32 [n, ceil(2k / 32)] packed k-mers"""
    n, k = c.shape
    wpt = (2 * k + 31) // 32
    c = np.concatenate([c.astype(np.uint32), np.zeros((n, wpt * 16 - k), np.uint32)], axis=1).reshape(n, wpt, 16)
    return (c << (2 * np.arange(15, -1, -1, dtype=np.uint32))).sum(axis=2, dtype=np.uint32)


def unpack_chars(words, k):
    w = np.asarray(words, np.uint32)
    return ((w[:, :, None] >> (2 * np.arange(15, -1, -1, dtype=np.uint32))) & 3).reshape(len(w), -1)[:, :k].astype(np.uint8)


def strings(chars):
    return [r.tobytes().decode() for r in ACGT[chars]]


class Restated:
    def __init__(self, sec, k):
        self.k = k
        self.wpt = wpt = (2 * k + 31) // 32
        size = self.size = int(np.frombuffer(sec["hdr"], np.int64)[0])
        w = np.frombuffer(sec["w"], "<u8")
        self.W = W = ((w[:, None] >> (4 * np.arange(16, dtype=np.uint64))) & 15).reshape(-1)[:size].astype(np.int64)
        self.last, self.tip, self.invalid = (_bits(sec[s], size) for s in ("last", "is_tip", "invalid"))
        self.f = np.frombuffer(sec["f"], np.int64)
        self.rank_f = np.frombuffer(sec["rank_f"], np.int64)
        self.mult = None
        if "edge_multi" in sec:
            self.mult = np.frombuffer(sec["edge_multi"], np.uint8).astype(np.int64)
            lg = np.frombuffer(sec["large_multi"], np.int64).reshape(-1, 2)
            self.mult[lg[:, 0]] = lg[:, 1]
        ts = np.frombuffer(sec["tip_seq"], "<u4").reshape(-1, wpt)
        self.tip_chars = unpack_chars(ts, k - 1) if k > 1 else np.zeros((len(ts), 0), np.uint8)   # [t, s]: s = 0 is the last character
        idx = np.arange(size)
        self.last_pos = np.flatnonzero(self.last)
        self.node = np.concatenate([[0], np.cumsum(self.last)])[:size]              # real nodes before edge i
        self.tip_idx = np.concatenate([[0], np.cumsum(self.tip)])[:size]
        self.lastc = np.searchsorted(self.f[1:5], idx, side="right")                 # 1..4
        # FORWARD: the target of the unflagged c edge number r is real node rank_f[c] + r
        a = np.where(W > 4, W - 4, W)
        fwd = np.full(size, -1, np.int64)
        self.unflagged_pos = {}
        for c in range(1, 5):
            pos = np.flatnonzero(W == c)
            self.unflagged_pos[c] = pos
            sel = a == c
            r = np.searchsorted(pos, idx[sel], side="right") - 1                     # the unflagged c edge at or before i
            fwd[sel] = self.last_pos[self.rank_f[c] + r]
        self.fwd = fwd
        # BACKWARD
        bwd = np.full(size, -1, np.int64)
        real = ~self.tip
        for c in range(1, 5):
            sel = real & (self.lastc == c)
            bwd[sel] = self.unflagged_pos[c][self.node[sel] - self.rank_f[c]]
        self.bwd = bwd
        # LABEL: walk BACKWARD, finish from a stored tip label
        lab = np.zeros((size, k), np.uint8)
        tipflag = self.tip.astype(np.uint32)
        t = self.tip_chars[self.tip_idx[self.tip]]
        lab[self.tip, 1:] = t[:, ::-1]
        e = idx[real]
        rows = idx[real]
        for p in range(k - 1, -1, -1):
            lab[rows, p] = self.lastc[e] - 1
            if p == 0:
                break
            e = bwd[e]
            at_tip = self.tip[e]
            if at_tip.any():
                tc = self.tip_chars[self.tip_idx[e[at_tip]]]                         # chars p-1-s = s-th stored character
                lab[rows[at_tip], :p] = tc[:, :p][:, ::-1]
                rows, e = rows[~at_tip], e[~at_tip]
        self.lab, self.tipflag = lab, tipflag
        # nodes: edges up to and including the node's last = 1 edge; valid out-edges in edge order
        nn = len(self.last_pos)
        valid = ~self.invalid
        out_tab = np.full((nn + 1, 4), -1, np.int64)
        ve = idx[valid]
        vn = self.node[ve]
        slot = np.arange(len(ve)) - np.searchsorted(vn, vn, side="left")
        out_tab[vn, slot] = ve
        self.out_tab = out_tab
        # incoming: every valid edge listed under the real node FORWARD leads to, in edge order
        in_tab = np.full((nn + 1, 4), -1, np.int64)
        tn = self.node[self.fwd[ve]]
        order = np.argsort(tn, kind="stable")
        tn_s, ve_s = tn[order], ve[order]
        slot = np.arange(len(ve_s)) - np.searchsorted(tn_s, tn_s, side="left")
        in_tab[tn_s, slot] = ve_s
        self.in_tab = in_tab
        # LOOKUP: the label of every real node's last edge
        self.node_index = {lab[e].tobytes(): int(e) for e in self.last_pos}
        # REVCOMP: the (k+1)-mer of every valid edge
        ek = np.concatenate([lab, ((np.where(W > 4, W - 4, W) - 1) & 3)[:, None].astype(np.uint8)], axis=1)
        self.edge_kmers = ek
        self.edge_index = {ek[e].tobytes(): int(e) for e in ve}

    def run(self, op, x):
        """the result array the device query returns for input rows x"""
        if op == SQ_LOOKUP:
            chars = unpack_chars(x, self.k)
            return np.array([self.node_index.get(r.tobytes(), -1) for r in chars], np.int64)
        i = np.asarray(x, np.int64)
        real = ~self.tip[i]
        if op == SQ_LABEL:
            return np.concatenate([pack_chars(self.lab[i]), self.tipflag[i][:, None]], axis=1)
        if op == SQ_FORWARD:
            return self.fwd[i]
        if op == SQ_BACKWARD:
            return self.bwd[i]
        if op in (SQ_OUTGOING, SQ_INCOMING, SQ_OUTDEGREE, SQ_INDEGREE):
            tab = self.out_tab if op in (SQ_OUTGOING, SQ_OUTDEGREE) else self.in_tab
            r = np.where(real[:, None], tab[self.node[i]], -1)
            return r if op in (SQ_OUTGOING, SQ_INCOMING) else (r >= 0).sum(axis=1).astype(np.int64)
        if op == SQ_MULTIPLICITY:
            return self.mult[i]
        if op == SQ_REVCOMP:
            rc = (3 - self.edge_kmers[i])[:, ::-1]
            ok = ~self.invalid[i]
            return np.array([self.edge_index.get(r.tobytes(), -1) if o else -1 for r, o in zip(rc, ok)], np.int64)
        raise ValueError(op)


def brute_graph(rd, k, m, is_solid, n_short=None):
    """-> {(k+1)-mer bytes (characters 0..3, forward orientation): multiplicity} from every solid position of every read.
    Reads are held reversed, so the edge at offset o of a read R is reverse(R[o .. o + k]); assist reads (index >= n_short)
    and every position when m = 1 are solid; each occurrence also counts for the reverse complement (once for a
    palindrome), and a multiplicity stops at 65535."""
    n_short = rd["n_reads"] if n_short is None else n_short
    start = rd["start"].astype(np.int64)
    bases = O.unpack_stream(rd["seq"], int(start[-1]))
    nk1 = rd["max_len"] - k
    occ = {}
    for r in range(rd["n_reads"]):
        s0, L = int(start[r]), int(start[r + 1] - start[r])
        if L < k + 1:
            continue
        o = np.arange(L - k)
        if m > 1 and r < n_short:
            bit = r * nk1 + o
            o = o[(is_solid[bit >> 3] >> (bit & 7)) & 1 == 1]
        if not len(o):
            continue
        e = bases[s0 + o[:, None] + np.arange(k + 1)[None, :]][:, ::-1]
        for row in np.ascontiguousarray(e):
            key = row.tobytes()
            occ[key] = occ.get(key, 0) + 1
    edges = {}
    for key, n in occ.items():
        rc = (3 - np.frombuffer(key, np.uint8))[::-1].tobytes()
        for x in {key, rc}:
            edges[x] = min(65535, edges.get(x, 0) + n)
    return edges
