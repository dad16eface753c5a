// sdbg_nav.cuh -- BOSS navigation on the device SdBG, shared by the batched queries (sdbg_query.cu) and the unitig
// builder (sdbg_unitig.cu): the rank / select chains over the tables sdbg_index.cu built, and the host code that points a
// QueryParams at a finished mgta_sdbg.
//
// Every step is a rank or a select on the W / last / is_tip tables (major every 65536, minor every 256, select samples
// every 256th occurrence, in-word nibble / bit counts).  Node boundaries come from `last`: the edges of a real node are
// the ones after the previous last = 1 edge up to its own last = 1 edge.  Tip edges have last = 0 (they sort in front of
// the real nodes of their group), so such a range may start with tip edges of other nodes; every node-level function
// skips them, and a tip edge's own node ($ + k - 1 characters) has no valid edges.  LOOKUP is a binary search in edge
// order (compare_node), not the BOSS forward search: see there.
#pragma once
#include <stdlib.h>
#include <string.h>

#include "sdbg_index.cuh"

namespace mgta_sdbg_impl {

constexpr int MAX_WPT = (2 * MGTA_MAX_K + 31) / 32;
constexpr unsigned long long NIB1 = 0x1111111111111111ull;

struct QueryParams {
    const unsigned long long *w, *last, *tip, *invalid;
    const uint8_t *edge_multi;
    const unsigned long long *large_edge;
    const uint16_t *large_val;
    const uint32_t *tip_seq;
    const uint16_t *w_minor, *last_minor, *tip_minor;
    const long long *w_major, *last_major, *tip_major;
    const uint32_t *w_sel[9], *last_sel;
    const long long *bucket_start;     // first edge of every lv1 bucket; null: LOOKUP starts from the f blocks
    long long size, n_minor, n_major, n_large, last_ones, tip_ones;
    long long w_freq[9], f[6], rank_f[6];
    int k, wpt;
    const void *in;
    void *out;
    unsigned long long n, row0;        // rows of this launch, global index of its first row
    unsigned long long *bad_row;       // atomicMin of the global index of every row with an edge id outside [0, size)
};

// nibble j of x equal to c -> bit 4 j of the result
__device__ __forceinline__ unsigned long long match_char(unsigned long long x, unsigned c) {
    x ^= ~(NIB1 * c);
    x &= x >> 2;
    x &= x >> 1;
    return x & NIB1;
}

__device__ __forceinline__ int get_w(const QueryParams &P, long long i) { return (int)((P.w[i >> 4] >> ((i & 15) * 4)) & 15ull); }
__device__ __forceinline__ bool get_bit(const unsigned long long *v, long long i) { return (v[i >> 6] >> (i & 63)) & 1ull; }

// occurrences of character c (1..8) in W[0, pos)
__device__ inline long long rank_w(const QueryParams &P, int c, long long pos) {
    if (pos <= 0) return 0;
    if (pos >= P.size) return P.w_freq[c];
    const long long iv = pos / 256;
    long long r = P.w_major[c * P.n_major + iv / 256] + (long long)P.w_minor[c * P.n_minor + iv];
    for (long long q = iv * 256; q < pos; q += 16) {
        unsigned long long m = match_char(P.w[q / 16], (unsigned)c);
        if (pos - q < 16) m &= (1ull << (4 * (pos - q))) - 1ull;
        r += __popcll(m);
    }
    return r;
}

__device__ __forceinline__ long long rank_last(const QueryParams &P, long long pos) {
    return rank1(P.last, P.last_minor, P.last_major, P.size, P.last_ones, pos);
}
__device__ __forceinline__ long long rank_tip(const QueryParams &P, long long pos) {
    return rank1(P.tip, P.tip_minor, P.tip_major, P.size, P.tip_ones, pos);
}

// the 256-position interval that holds occurrence r (0-based): the sample brackets it, a binary search over the
// exclusive counts Occ(i) = major[i / 256] + minor[i] finds the last interval with Occ(i) <= r
__device__ __forceinline__ long long select_interval(const uint32_t *sel, const uint16_t *minor, const long long *major, long long r,
                                                     long long *occ) {
    long long lo = sel[r / 256], hi = sel[r / 256 + 1];
    while (lo < hi) {
        const long long mid = (lo + hi + 1) >> 1;
        if (major[mid / 256] + (long long)minor[mid] <= r) lo = mid; else hi = mid - 1;
    }
    *occ = major[lo / 256] + (long long)minor[lo];
    return lo;
}

// position of occurrence r (0-based) of character c (1..8) in W, or -1
__device__ inline long long select_w(const QueryParams &P, int c, long long r) {
    if (r < 0 || r >= P.w_freq[c]) return -1;
    long long occ;
    const long long iv = select_interval(P.w_sel[c], P.w_minor + c * P.n_minor, P.w_major + c * P.n_major, r, &occ);
    long long need = r - occ;
    for (long long wi = iv * 16; wi < iv * 16 + 16; ++wi) {
        unsigned long long m = match_char(P.w[wi], (unsigned)c);
        const int cnt = __popcll(m);
        if (need < cnt) {
            for (; need > 0; --need) m &= m - 1;
            return wi * 16 + (__ffsll((long long)m) - 1) / 4;
        }
        need -= cnt;
    }
    return -1;
}

// position of the one number r (0-based) of `last`, or -1
__device__ inline long long select_last(const QueryParams &P, long long r) {
    if (r < 0 || r >= P.last_ones) return -1;
    long long occ;
    const long long iv = select_interval(P.last_sel, P.last_minor, P.last_major, r, &occ);
    long long need = r - occ;
    for (long long wi = iv * 4; wi < iv * 4 + 4; ++wi) {
        unsigned long long x = P.last[wi];
        const int cnt = __popcll(x);
        if (need < cnt) {
            for (; need > 0; --need) x &= x - 1;
            return wi * 64 + __ffsll((long long)x) - 1;
        }
        need -= cnt;
    }
    return -1;
}

// last character (1..4) of v(i): the f block that holds i
__device__ __forceinline__ int last_char_of(const QueryParams &P, long long i) {
    int c = 4;
    while (c > 1 && i < P.f[c]) --c;
    return c;
}

__device__ inline long long forward(const QueryParams &P, long long i) {
    int a = get_w(P, i);
    if (a == 0) return -1;
    if (a > 4) a -= 4;
    return select_last(P, P.rank_f[a] + rank_w(P, a, i + 1) - 1);
}

__device__ inline long long backward(const QueryParams &P, long long i) {
    if (get_bit(P.tip, i)) return -1;
    const int c = last_char_of(P, i);
    return select_w(P, c, rank_last(P, i) - P.rank_f[c]);
}

// character t of the stored label of tip edge e: t = 0 is the node's last character (the record's key order)
__device__ __forceinline__ unsigned tip_char(const QueryParams &P, long long tip_idx, int t) {
    return (P.tip_seq[tip_idx * P.wpt + (t >> 4)] >> (2 * (15 - (t & 15)))) & 3u;
}

__device__ __forceinline__ unsigned kmer_char(const uint32_t *x, int u) { return (x[u >> 4] >> (2 * (15 - (u & 15)))) & 3u; }
__device__ __forceinline__ void put_char(uint32_t *x, int u, unsigned c) { x[u >> 4] |= c << (2 * (15 - (u & 15))); }

// the k characters of v(i) in forward orientation; returns 1 for a tip node (its '$' stays 0)
__device__ inline int label(const QueryParams &P, long long i, uint32_t *x) {
    for (int j = 0; j < P.wpt; ++j) x[j] = 0;
    long long e = i;
    int p = P.k - 1;
    if (get_bit(P.tip, e)) {
        const long long t = rank_tip(P, e);
        for (int s = 0; s + 1 < P.k; ++s) put_char(x, P.k - 1 - s, tip_char(P, t, s));
        return 1;
    }
    while (true) {                                                  // v(e) ends at character p of the label
        put_char(x, p, (unsigned)last_char_of(P, e) - 1u);
        if (p == 0 || (e = backward(P, e)) < 0) break;
        --p;
        if (get_bit(P.tip, e)) {                                   // the rest is the tail of a stored tip label
            const long long t = rank_tip(P, e);
            for (int s = 0; s <= p; ++s) put_char(x, p - s, tip_char(P, t, s));
            break;
        }
    }
    return 0;
}

// colex order of v(e) against the query k-mer x: the characters from the last one backwards, '$' before A (the order of
// the edges).  Character d of v(e) from the end is the last character of BACKWARD^d(e); once the walk reaches a tip edge
// the rest comes from its stored label.  -> < 0, 0, > 0
__device__ inline int compare_node(const QueryParams &P, long long e, const uint32_t *x) {
    bool tip = get_bit(P.tip, e);
    long long t = tip ? rank_tip(P, e) : 0;
    int base = 0;                                                  // depth at which the walk reached the tip node
    for (int d = 0; d < P.k; ++d) {
        const int xc = (int)kmer_char(x, P.k - 1 - d);
        const int s = d - base;
        const int ce = tip ? (s == P.k - 1 ? -1 : (int)tip_char(P, t, s)) : last_char_of(P, e) - 1;
        if (ce != xc) return ce < xc ? -1 : 1;
        if (!tip && d + 1 < P.k) {
            e = backward(P, e);
            if (e < 0) return -1;
            if (get_bit(P.tip, e)) { tip = true; t = rank_tip(P, e); base = d + 1; }
        }
    }
    return 0;
}

// IndexBinarySearch: the first edge whose node is not below x in edge order, inside the lv1 bucket of x's last 8
// characters (or the f block of its last character).  The textbook BOSS forward search (two ranks per character) needs a
// node for every prefix of x; this SdBG keeps only one-'$' tip nodes, so near a read start those prefixes have no node.
__device__ inline long long lookup(const QueryParams &P, const uint32_t *x) {
    long long lo, hi;
    if (P.bucket_start && P.k > 8) {                               // lv1 bucket = the node's last 8 characters, last first
        unsigned b = 0;
        for (int t = 0; t < 8; ++t) b |= kmer_char(x, P.k - 1 - t) << (2 * (7 - t));
        lo = P.bucket_start[b]; hi = P.bucket_start[b + 1];
    } else {
        const int c = (int)kmer_char(x, P.k - 1) + 1;
        lo = P.f[c]; hi = c < 4 ? P.f[c + 1] : P.size;
    }
    const long long end = hi;
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (compare_node(P, mid, x) < 0) lo = mid + 1; else hi = mid;
    }
    if (lo >= end || compare_node(P, lo, x) != 0) return -1;
    return select_last(P, rank_last(P, lo));
}

// edges of the real node v(i): [first, last]
__device__ __forceinline__ void node_edges(const QueryParams &P, long long i, long long *first, long long *last) {
    const long long r = rank_last(P, i);
    *first = r == 0 ? 0 : select_last(P, r - 1) + 1;
    *last = select_last(P, r);
}

__device__ inline int outgoing(const QueryParams &P, long long i, long long *out) {
    int n = 0;
    if (get_bit(P.tip, i)) return 0;
    long long a, b;
    node_edges(P, i, &a, &b);
    for (long long e = a; e <= b && n < 4; ++e)
        if (!get_bit(P.invalid, e)) out[n++] = e;
    return n;
}

// the unflagged edge into v(i), then the flagged edges with the same character up to the next unflagged one
__device__ inline int incoming(const QueryParams &P, long long i, long long *out) {
    int n = 0;
    const long long b = backward(P, i);
    if (b < 0) return 0;
    const int c = get_w(P, b);
    const long long rb = rank_w(P, c, b + 1);
    const long long next = rb < P.w_freq[c] ? select_w(P, c, rb) : P.size;
    if (!get_bit(P.invalid, b)) out[n++] = b;
    const long long f1 = rank_w(P, c + 4, next);
    for (long long r = rank_w(P, c + 4, b + 1); r < f1 && n < 4; ++r) out[n++] = select_w(P, c + 4, r);
    return n;
}

__device__ inline long long multiplicity(const QueryParams &P, long long i) {
    const int m = P.edge_multi[i];
    if (m < 255) return m;
    long long lo = 0, hi = P.n_large - 1;
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if ((long long)P.large_edge[mid] < i) lo = mid + 1; else hi = mid;
    }
    return P.n_large > 0 && (long long)P.large_edge[lo] == i ? (long long)P.large_val[lo] : -1;
}

__device__ inline long long revcomp(const QueryParams &P, long long i) {
    if (get_bit(P.invalid, i)) return -1;
    uint32_t x[MAX_WPT], y[MAX_WPT];
    label(P, i, x);
    const unsigned a = (unsigned)(get_w(P, i) - 1) & 3u, want = 3u - kmer_char(x, 0);
    for (int j = 0; j < P.wpt; ++j) y[j] = 0;                     // reverse complement of x.a, without its last character
    put_char(y, 0, 3u - a);
    for (int j = 1; j < P.k; ++j) put_char(y, j, 3u - kmer_char(x, P.k - j));
    const long long l = lookup(P, y);
    if (l < 0) return -1;
    const long long r = rank_last(P, l);
    for (long long e = r == 0 ? 0 : select_last(P, r - 1) + 1; e <= l; ++e) {
        const int we = get_w(P, e);
        if (we != 0 && !get_bit(P.tip, e) && ((unsigned)(we - 1) & 3u) == want) return e;
    }
    return -1;
}

inline bool on_device(const void *p) {
    cudaPointerAttributes pa;
    const bool d = cudaPointerGetAttributes(&pa, p) == cudaSuccess && pa.type == cudaMemoryTypeDevice;
    cudaGetLastError();
    return d;
}

inline long long env_ll(const char *name, long long dflt) {
    const char *s = getenv(name);
    return s && *s ? atoll(s) : dflt;
}

// points P at the arrays and tables of the finished graph g; the first call uploads the lv1 bucket starts for LOOKUP.
// The per-launch fields (in, out, n, row0, bad_row) stay zero.
inline int query_params(mgta_sdbg *g, QueryParams *out) {
    int rc;
    if (!g->q_bucket.cap) {                                        // first use: the lv1 bucket offsets to the device
        if ((rc = grow(g, g->q_bucket, g->bucket_start.size() * 8, 0))) return rc;
        SCK(cudaMemcpyAsync(g->q_bucket.p, g->bucket_start.data(), g->bucket_start.size() * 8, cudaMemcpyHostToDevice, g->stream));
    }
    QueryParams &P = *out;
    memset(&P, 0, sizeof(P));
    P.w = (const unsigned long long *)g->w.p; P.last = (const unsigned long long *)g->last.p; P.tip = (const unsigned long long *)g->tip.p;
    P.invalid = (const unsigned long long *)g->invalid.p; P.edge_multi = (const uint8_t *)g->edge_multi.p;
    P.large_edge = (const unsigned long long *)g->large_edge.p; P.large_val = (const uint16_t *)g->large_val.p;
    P.tip_seq = (const uint32_t *)g->tip_seq.p;
    P.w_minor = (const uint16_t *)g->w_minor.p; P.last_minor = (const uint16_t *)g->last_minor.p; P.tip_minor = (const uint16_t *)g->tip_minor.p;
    P.w_major = (const long long *)g->w_major.p; P.last_major = (const long long *)g->last_major.p; P.tip_major = (const long long *)g->tip_major.p;
    for (int c = 0; c < 9; ++c) { P.w_sel[c] = (const uint32_t *)g->w_sel[c].p; P.w_freq[c] = g->w_freq[c]; }
    P.last_sel = (const uint32_t *)g->last_sel.p;
    P.bucket_start = (const long long *)g->q_bucket.p;
    P.size = g->n_edges; P.n_minor = g->n_minor; P.n_major = g->n_major; P.n_large = g->need_mult ? g->n_large : 0;
    P.last_ones = g->last_ones; P.tip_ones = g->tip_ones;
    for (int j = 0; j < 6; ++j) { P.f[j] = g->f[j]; P.rank_f[j] = g->rank_f[j]; }
    P.k = g->kmer_k; P.wpt = g->wpt;
    return MGTA_OK;
}

}  // namespace mgta_sdbg_impl
