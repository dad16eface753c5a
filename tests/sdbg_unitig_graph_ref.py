"""TEST INFRASTRUCTURE ONLY: the links of include/mgta_sdbg_unitig_graph.h from the unitig rows and strings alone.

`string_links(rows, seq, k)` returns the exact array the device returns.  It uses no edge id and no navigation: a link
a -> b is there exactly when the last k characters of oriented unitig a equal the first k of b, and a cycle row links
to itself.  tests/test_sdbg_unitig_graph_cpu.py pins it against an edge-level restatement of the header's definition.
"""
import numpy as np

from sdbg_unitig_ref import CYCLE, SELF_RC, read_dict


def _rc(s):
    return s[::-1].translate(str.maketrans("ACGT", "TGCA"))


def bar(rows, o):
    """the reverse orientation of oriented unitig o"""
    return o if rows[o >> 1, 5] & SELF_RC else o ^ 1


def all_string_links(rows, seq, k):
    """the full link set F: a set of (a, b), closed under the twin map"""
    rows = np.asarray(rows)
    b = bytes(np.asarray(seq, np.uint8))
    ends = np.append(rows[1:, 3], len(b)) if len(rows) else np.zeros(0, np.int64)
    oriented, F = {}, set()
    for r, (row, end) in enumerate(zip(rows.tolist(), ends.tolist())):
        s = b[row[3]:end].decode()
        if row[5] & CYCLE:
            F.add((2 * r, 2 * r))
            F.add((bar(rows, 2 * r), bar(rows, 2 * r)))
            continue
        oriented[2 * r] = s
        if not row[5] & SELF_RC:
            oriented[2 * r + 1] = _rc(s)
    by_prefix = {}
    for o, s in oriented.items():
        by_prefix.setdefault(s[:k], []).append(o)
    for a, s in oriented.items():
        for o in by_prefix.get(s[-k:], ()):
            F.add((a, o))
    return F


def canonical_links(rows, F):
    """the pairs (a, b) of F with (a, b) <= (bar(b), bar(a)), sorted -> int64 [L, 2]"""
    rows = np.asarray(rows)
    out = sorted((a, b) for a, b in F if (a, b) <= (bar(rows, b), bar(rows, a)))
    return np.array(out, np.int64).reshape(-1, 2)


def string_links(rows, seq, k):
    """-> int64 [L, 2]: the canonical links (from, to), sorted, as Sdbg.unitig_links returns them"""
    return canonical_links(rows, all_string_links(rows, seq, k))


def hairpins(rows, links):
    """links a -> bar(a)"""
    return [(a, b) for a, b in np.asarray(links).tolist() if b == bar(np.asarray(rows), a) and not rows[a >> 1, 5] & CYCLE]


# ---- a seeded read set with hairpins -------------------------------------------------------------------------------------
def hairpin_reads(seed=4, k=16, flanks=5, flank_len=40, core=40):
    """reads through a palindromic k-mer P and through a palindrome C of `core` characters, each between `flanks` random
    left and right flanks, on both strands.  P is a node with several in- and out-edges, so the unitig that ends on P
    links to its own reverse complement (a hairpin, at even k only); C's middle is a linear unitig that is its own
    reverse complement, with links at both ends."""
    rng = np.random.default_rng(seed)
    h = rng.integers(0, 4, size=k // 2, dtype=np.uint8)
    P = np.concatenate([h, (3 - h)[::-1]])
    c = rng.integers(0, 4, size=core // 2, dtype=np.uint8)
    C = np.concatenate([c, (3 - c)[::-1]])
    reads = []
    for mid in (P, C):
        for _ in range(flanks):
            r = np.concatenate([rng.integers(0, 4, size=flank_len, dtype=np.uint8), mid, rng.integers(0, 4, size=flank_len, dtype=np.uint8)])
            reads += [r, (3 - r)[::-1]]
    return read_dict(reads)
