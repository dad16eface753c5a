"""TEST INFRASTRUCTURE ONLY: two checkers for the unitigs of include/mgta_sdbg_unitig.h.

- `restated_unitigs(ref)`: the exact rows and sequence bytes the device returns, from a `Restated` graph
  (tests/sdbg_query_ref.py): succ from its out / in tables, the unitigs by walking every head in lockstep and then every
  leftover cycle from its smallest edge.  No rulers, no list ranking: it shares no logic with megagta_b200/csrc/sdbg_unitig.cu.
- `brute_unitigs(E, k)`: the unitigs compacted straight from the (k+1)-mer strings of `brute_graph`, canonical per
  reverse-complement pair.
"""
from collections import Counter

import numpy as np

import sdbg_query_ref as R

ACGT = np.frombuffer(b"ACGT", np.uint8)
CYCLE, SELF_RC = 1, 2


def restated_unitigs(ref):
    """-> (rows int64 [U, 6]: first_edge, last_edge, n_edges, seq_offset, mult_sum, flags; seq uint8 [chars])"""
    size, k = ref.size, ref.k
    ve = np.flatnonzero(~ref.invalid)
    outdeg = (ref.out_tab >= 0).sum(axis=1)
    indeg = (ref.in_tab >= 0).sum(axis=1)
    succ = np.full(size, -1, np.int64)
    t = ref.node[ref.fwd[ve]]
    one = (outdeg[t] == 1) & (indeg[t] == 1)
    succ[ve[one]] = ref.out_tab[t[one], 0]
    has_pred = np.zeros(size, bool)
    has_pred[succ[succ >= 0]] = True
    head = np.full(size, -1, np.int64)
    pos = np.full(size, -1, np.int64)
    cur = ve[~has_pred[ve]]                                        # linear unitigs: all heads one step at a time
    owner, p = cur.copy(), 0
    while len(cur):
        head[cur], pos[cur] = owner, p
        nxt = succ[cur]
        cur, owner, p = nxt[nxt >= 0], owner[nxt >= 0], p + 1
    cycle = set()
    for e in ve[head[ve] < 0].tolist():                            # ascending: the first edge met of a cycle is its smallest
        if head[e] >= 0:
            continue
        x, p = e, 0
        while True:
            head[x], pos[x] = e, p
            x, p = int(succ[x]), p + 1
            if x == e:
                break
        cycle.add(e)
    e1, n = np.unique(head[ve], return_counts=True)
    n_of = dict(zip(e1.tolist(), n.tolist()))
    last = np.zeros(size, np.int64)
    is_last = pos[ve] == np.array([n_of[h] for h in head[ve].tolist()]) - 1
    last[head[ve[is_last]]] = ve[is_last]
    last = last[e1]
    mult = np.full(len(e1), -1, np.int64)
    if ref.mult is not None:
        idx = np.searchsorted(e1, head[ve])
        mult = np.bincount(idx, weights=ref.mult[ve], minlength=len(e1)).astype(np.int64)
    rc = ref.run(R.SQ_REVCOMP, last)
    partner = np.where(rc >= 0, head[np.maximum(rc, 0)], e1)
    keep = e1 <= partner
    flags = np.array([CYCLE if e in cycle else 0 for e in e1.tolist()], np.int64) | np.where((partner == e1) & (rc >= 0), SELF_RC, 0)
    order = ve[np.lexsort((pos[ve], head[ve]))]                   # grouped by e1, in path order
    start = np.concatenate([[0], np.cumsum(n)])
    wc = ((ref.W - 1) & 3).astype(np.uint8)
    pieces = []
    for j in np.flatnonzero(keep).tolist():
        pieces += [ref.lab[e1[j]], wc[order[start[j]:start[j + 1]]]]
    seq = ACGT[np.concatenate(pieces)] if pieces else np.zeros(0, np.uint8)
    kn = k + n[keep]
    rows = np.stack([e1[keep], last[keep], n[keep], np.concatenate([[0], np.cumsum(kn)[:-1]]).astype(np.int64), mult[keep],
                     flags[keep]], axis=1).astype(np.int64) if keep.any() else np.zeros((0, 6), np.int64)
    return rows, seq


def _rc(s):
    return s[::-1].translate(str.maketrans("ACGT", "TGCA"))


def _least_rotation(w):
    return min(w[i:] + w[:i] for i in range(len(w)))


def canonical(seq, k, cycle):
    """a linear unitig -> min(s, revcomp(s)); a cycle -> the least rotation, over both strands, of its n-character cyclic
    word (the characters after the first k)"""
    if cycle:
        w = seq[k:]
        return min(_least_rotation(w), _least_rotation(_rc(w)))
    return min(seq, _rc(seq))


def brute_unitigs(E, k):
    """{(k+1)-mer bytes: multiplicity} -> Counter of (cycle, self reverse complement, canonical string, multiplicity sum),
    one entry per reverse-complement pair"""
    out, indeg = {}, Counter()
    for e in E:
        out.setdefault(e[:k], []).append(e)
        indeg[e[1:]] += 1

    def simple(node):
        return indeg[node] == 1 and len(out.get(node, ())) == 1

    def succ(e):
        return out[e[1:]][0] if simple(e[1:]) else None

    def rc(e):
        return (3 - np.frombuffer(e, np.uint8))[::-1].tobytes()

    seen, res = set(), Counter()

    def add(path, cycle):
        s = "".join("ACGT"[c] for c in path[0]) + "".join("ACGT"[p[k]] for p in path[1:])
        mirror = [rc(e) for e in path]
        self_rc = set(mirror) == set(path)
        seen.update(path)
        seen.update(mirror)
        res[(cycle, self_rc, canonical(s, k, cycle), sum(E[e] for e in path))] += 1

    for e in sorted(E):
        if e in seen or simple(e[:k]):
            continue
        path = [e]
        while (x := succ(path[-1])) is not None:
            path.append(x)
        add(path, False)
    for e in sorted(E):                                            # what is left lies on cycles
        if e in seen:
            continue
        path = [e]
        while (x := succ(path[-1])) != e:
            path.append(x)
        add(path, True)
    return res


def canonical_rows(rows, seq, k, with_mult=True):
    """device or restated rows -> the Counter brute_unitigs returns (mult_sum left out when with_mult is False)"""
    b = bytes(np.asarray(seq, np.uint8))
    ends = np.append(rows[1:, 3], len(b))
    return Counter((bool(r[5] & CYCLE), bool(r[5] & SELF_RC), canonical(b[r[3]:end].decode(), k, bool(r[5] & CYCLE)),
                    int(r[4]) if with_mult else None) for r, end in zip(rows.tolist(), ends.tolist()))


def edge_invariant(rows):
    """sum of n_edges, twice for a unitig that is not its own reverse complement: the number of valid edges"""
    return int((rows[:, 2] * np.where(rows[:, 5] & SELF_RC, 1, 2)).sum())


# ---- seeded read sets for the hard shapes -------------------------------------------------------------------------------
def read_dict(reads):
    """uint8 arrays of bases 0..3 -> the read dict oracle.load_read_lib returns"""
    from oracle import oracle as O
    lens = np.array([len(r) for r in reads], np.int64)
    start = np.zeros(len(reads) + 1, np.uint64)
    start[1:] = np.cumsum(lens)
    seq, start = O.pack_reversed(np.concatenate(reads).astype(np.uint8), start)
    return dict(seq=seq, start=start, n_reads=len(reads), max_len=int(lens.max()))


def _tile(rng, g, read_len, step):
    """error-free reads of g every `step` bases, each on a random strand"""
    out = []
    for p in range(0, len(g) - read_len + 1, step):
        r = g[p:p + read_len]
        out.append(r if rng.integers(2) else (3 - r)[::-1])
    return out


def long_genome_reads(seed=1, genome=200_000, read_len=150, step=50):
    """one random genome: a unitig of about `genome` edges and its reverse complement"""
    rng = np.random.default_rng(seed)
    g = rng.integers(0, 4, size=genome, dtype=np.uint8)
    return read_dict(_tile(rng, g, read_len, step))


def circular_genome_reads(seed=2, genome=5000, read_len=150, step=40):
    """reads of a circular genome, some across the origin: a cycle of `genome` edges and its reverse complement, plus one
    unrelated read (Restated needs at least one tip node)"""
    rng = np.random.default_rng(seed)
    g = rng.integers(0, 4, size=genome, dtype=np.uint8)
    extra = rng.integers(0, 4, size=read_len, dtype=np.uint8)
    return read_dict(_tile(rng, np.concatenate([g, g[:read_len + step]]), read_len, step) + [extra])


def tandem_reads(seed=3, read_len=120, units=("A", "AC", "AACGT", "ACCGATT", "AGCTTGACCATGA")):
    """reads that are pure tandem repeats of short units (a cycle of len(unit) edges each, poly-A a self-loop) on both
    strands, and a few random reads"""
    rng = np.random.default_rng(seed)
    reads = []
    for u in units:
        rep = np.tile(np.array(["ACGT".index(c) for c in u], np.uint8), read_len // len(u) + 1)[:read_len]
        reads += [rep, (3 - rep)[::-1]]
    reads += [rng.integers(0, 4, size=read_len, dtype=np.uint8) for _ in range(6)]
    return read_dict(reads)
