// sdbg_unitig.cu -- the unitigs of the device SdBG (include/mgta_sdbg_unitig.h): every maximal non-branching path with its
// sequence and summed multiplicity, by list ranking in HBM.
//
// A unitig can be 10^5 edges long, so no thread walks a whole one.  The kernels, in order:
//   k_ut_links    one thread per edge: succ (-2 for an invalid edge, -1 for none) from the degrees of the target node,
//                 and has_pred[succ] = 1 (a plain store: a target with in-degree 1 has one writer)
//   k_ut_mark     rulers = heads (valid, no predecessor) + every valid edge whose hash falls in 1 / S of the range
//   scan          ruler ids in edge order (k_ut_scan_*: tile scan, one block over the tile sums, add)
//   k_ut_walk     one thread per ruler walks succ up to the next ruler: every edge gets its ruler and local offset, the
//                 segment its length, multiplicity, smallest edge and the next ruler.  Expected length S.
//   k_ut_resid    cycles short enough to hold no ruler are the valid edges left unvisited: the smallest edge of such a
//                 cycle (the one whose walk around it meets no smaller id) becomes a ruler, and k_ut_walk runs again
//   k_ut_jump_a   pointer jumping over the ruler predecessors with a min reduction: the rulers still pointing somewhere
//                 after ceil(log2 R) rounds lie on a cycle, and know its smallest edge; k_ut_break cuts every cycle in
//                 front of the ruler whose segment holds that edge
//   k_ut_jump_b   pointer jumping (Wyllie) over the now acyclic ruler lists: every ruler's root and prefix length /
//                 multiplicity; k_ut_tot gives each root the totals of its list
//   k_ut_place    every edge: its unitig's e1 and its offset (for a cycle modulo n, relative to the smallest edge)
//   k_ut_table    one thread per unitig: REVCOMP of its last edge decides whether it is kept; scan in edge order =
//                 row order; k_ut_rows writes the rows, a scan of k + n the sequence offsets
//   k_ut_scatter  every edge of a kept unitig writes its character; e1 also the k characters of LABEL(v(e1))
// Scratch is int64 per edge and per ruler (edge ids pass 2^32) and is freed before mgta_sdbg_unitigs returns.
//
// The links between the unitigs (include/mgta_sdbg_unitig_graph.h), over the rows of the last mgta_sdbg_unitigs:
//   k_ul_heads    one thread per row and side: id of every head (hid[first_edge] = 2r, hid[REVCOMP(last_edge)] = 2r + 1
//                 for the partner of a row that is not its own reverse complement) and the partner's end REVCOMP(first_edge)
//   k_ul_count    one thread per oriented unitig: FORWARD of its end, OUTGOING there, each out-edge through hid; counts
//                 the canonical links.  scan of the counts = the output offsets in `from` order; k_ul_write repeats the
//                 walk and writes the `to` values sorted inside the thread
// Scratch is int64 per edge (hid) and per oriented unitig, and is freed before mgta_sdbg_unitig_links returns.
#include "sdbg_nav.cuh"
#include "../../include/mgta_sdbg_unitig.h"
#include "../../include/mgta_sdbg_unitig_graph.h"

using namespace mgta_sdbg_impl;

namespace {

constexpr int TPB = 256;
constexpr int SCAN_PER = 8, SCAN_TILE = TPB * SCAN_PER;

#define FOR_EACH(i, n) for (long long i = blockIdx.x * (long long)TPB + threadIdx.x; i < (n); i += (long long)gridDim.x * TPB)

// one ruler: its segment (the ruler edge up to the edge before the next ruler) and, for a root, its unitig's totals
struct Seg {
    long long edge, next, prev;        // ruler edge, next / previous ruler in its unitig (-1: none)
    long long len, mult, mn, mnoff;    // edges, summed multiplicity, smallest edge id and its offset in the segment
    long long tot_len, tot_mult;       // roots only: totals of the unitig
    long long flags;                   // 1 = root of a cycle (cut in front of it), 2 = its own reverse complement, 4 = kept
};

unsigned grid_for(long long n) { return (unsigned)std::max(1ll, std::min((n + TPB - 1) / TPB, 148ll * 64)); }

__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {       // splitmix64 finaliser
    x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ull;
    x ^= x >> 27; x *= 0x94d049bb133111ebull;
    return x ^ (x >> 31);
}

__global__ void __launch_bounds__(TPB) k_ut_links(const QueryParams P, long long *succ, long long *rof, uint8_t *has_pred) {
    FOR_EACH(e, P.size) {
        rof[e] = -1;
        long long s = -2;
        if (!get_bit(P.invalid, e)) {
            const long long t = forward(P, e);
            long long o[4], in[4];
            s = outgoing(P, t, o) == 1 && incoming(P, t, in) == 1 ? o[0] : -1;
            if (s >= 0) has_pred[s] = 1;
        }
        succ[e] = s;
    }
}

__global__ void __launch_bounds__(TPB) k_ut_mark(long long n, const long long *succ, const uint8_t *has_pred, long long stride,
                                                 long long *is_ruler) {
    FOR_EACH(e, n) is_ruler[e] = succ[e] != -2 && (!has_pred[e] || mix64((unsigned long long)e) % (unsigned long long)stride == 0);
}

// ---- exclusive scan of int64 in place; x[n] receives the total ---------------------------------------------------------
__device__ __forceinline__ long long block_exclusive(long long v, long long *total) {
    __shared__ long long warp_sum[TPB / 32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    long long inc = v;
    for (int d = 1; d < 32; d <<= 1) {
        const long long u = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += u;
    }
    if (lane == 31) warp_sum[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        long long w = lane < TPB / 32 ? warp_sum[lane] : 0, wi = w;
        for (int d = 1; d < 32; d <<= 1) {
            const long long u = __shfl_up_sync(0xffffffffu, wi, d);
            if (lane >= d) wi += u;
        }
        if (lane < TPB / 32) warp_sum[lane] = wi - w;
        if (lane == TPB / 32 - 1) *total = wi;
    }
    __syncthreads();
    const long long r = warp_sum[wid] + inc - v;
    __syncthreads();
    return r;
}

__global__ void __launch_bounds__(TPB) k_ut_scan_tiles(long long *x, long long n, long long *tile_sum) {
    __shared__ long long total;
    const long long base = blockIdx.x * (long long)SCAN_TILE + threadIdx.x * (long long)SCAN_PER;
    long long v[SCAN_PER], s = 0;
    for (int j = 0; j < SCAN_PER; ++j) { v[j] = base + j < n ? x[base + j] : 0; s += v[j]; }
    long long run = block_exclusive(s, &total);
    for (int j = 0; j < SCAN_PER; ++j) {
        if (base + j < n) x[base + j] = run;
        run += v[j];
    }
    if (threadIdx.x == 0) tile_sum[blockIdx.x] = total;
}

// one block: exclusive scan of the tile sums in place, the grand total to *total
__global__ void __launch_bounds__(TPB) k_ut_scan_sums(long long *tile_sum, long long nt, long long *total) {
    __shared__ long long chunk_total;
    long long carry = 0;
    for (long long b = 0; b < nt; b += TPB) {
        const long long i = b + threadIdx.x;
        const long long v = i < nt ? tile_sum[i] : 0;
        const long long r = block_exclusive(v, &chunk_total);
        if (i < nt) tile_sum[i] = carry + r;
        __syncthreads();
        carry += chunk_total;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}

__global__ void __launch_bounds__(TPB) k_ut_scan_add(long long *x, long long n, const long long *tile_sum) {
    FOR_EACH(i, n) x[i] += tile_sum[i / SCAN_TILE];
}

int scan(mgta_sdbg *g, long long *x, long long n, long long *tile_sum) {
    const long long nt = (n + SCAN_TILE - 1) / SCAN_TILE;
    if (nt) k_ut_scan_tiles<<<(unsigned)nt, TPB, 0, g->stream>>>(x, n, tile_sum);
    k_ut_scan_sums<<<1, TPB, 0, g->stream>>>(tile_sum, nt, x + n);
    if (nt) k_ut_scan_add<<<grid_for(n), TPB, 0, g->stream>>>(x, n, tile_sum);
    SCK(cudaGetLastError());
    return MGTA_OK;
}

// ---- rulers and their segments ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(TPB) k_ut_rulers(long long n, const long long *ruler_id, Seg *seg, long long *rof) {
    FOR_EACH(e, n) if (ruler_id[e + 1] > ruler_id[e]) {
        seg[ruler_id[e]].edge = e;
        rof[e] = ruler_id[e];
    }
}

// rof of a ruler edge is set before the walk and rof of any other edge only by the one walk that reaches it (an edge has
// at most one predecessor), so rof[nx] >= 0 means that nx is a ruler
__global__ void __launch_bounds__(TPB) k_ut_walk(const QueryParams P, int need_mult, const long long *succ, long long *rof, long long *off,
                                                 Seg *seg, long long r0, long long r1) {
    FOR_EACH(j, r1 - r0) {
        const long long i = r0 + j, x = seg[i].edge;
        long long cur = x, len = 0, mult = 0, mn = x, mnoff = 0, next;
        while (true) {
            rof[cur] = i;
            off[cur] = len;
            if (need_mult) mult += multiplicity(P, cur);
            if (cur < mn) { mn = cur; mnoff = len; }
            ++len;
            const long long nx = succ[cur];
            if (nx < 0) { next = -1; break; }
            const long long r = rof[nx];
            if (r >= 0) { next = r; break; }
            cur = nx;
        }
        Seg &s = seg[i];
        s.next = next; s.prev = -1; s.len = len; s.mult = mult; s.mn = mn; s.mnoff = mnoff; s.flags = 0;
    }
}

__global__ void __launch_bounds__(TPB) k_ut_count_unvisited(long long n, const long long *succ, const long long *rof,
                                                            unsigned long long *count) {
    FOR_EACH(e, n) {
        const bool u = succ[e] != -2 && rof[e] < 0;
        const unsigned b = __ballot_sync(__activemask(), u);
        if (u && (threadIdx.x & 31) == __ffs(b) - 1) atomicAdd(count, (unsigned long long)__popc(b));
    }
}

// an unvisited valid edge lies on a cycle without a ruler; the smallest edge of that cycle becomes one
__global__ void __launch_bounds__(TPB) k_ut_resid(long long n, const long long *succ, long long *rof, Seg *seg,
                                                  unsigned long long *n_rulers) {
    FOR_EACH(x, n) if (succ[x] != -2 && rof[x] < 0) {
        long long y = succ[x];
        while (y > x) y = succ[y];
        if (y == x) {
            const long long i = (long long)atomicAdd(n_rulers, 1ull);
            seg[i].edge = x;
            rof[x] = i;
        }
    }
}

__global__ void __launch_bounds__(TPB) k_ut_prev(long long R, Seg *seg) {
    FOR_EACH(i, R) if (seg[i].next >= 0) seg[seg[i].next].prev = i;
}

// ---- list ranking over the rulers ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(TPB) k_ut_init_a(long long R, const Seg *seg, long long *p, long long *v) {
    FOR_EACH(i, R) { p[i] = seg[i].prev; v[i] = seg[i].mn; }
}

__global__ void __launch_bounds__(TPB) k_ut_jump_a(long long R, const long long *p, const long long *v, long long *p2, long long *v2) {
    FOR_EACH(i, R) {
        const long long q = p[i];
        p2[i] = q >= 0 ? p[q] : -1;
        v2[i] = q >= 0 ? min(v[i], v[q]) : v[i];
    }
}

// after the rounds of k_ut_jump_a p[i] >= 0 exactly on cycles, and v[i] is the cycle's smallest edge
__global__ void __launch_bounds__(TPB) k_ut_break(long long R, Seg *seg, const long long *p, const long long *v) {
    FOR_EACH(i, R) if (p[i] >= 0 && seg[i].mn == v[i]) { seg[i].prev = -1; seg[i].flags = 1; }
}

__global__ void __launch_bounds__(TPB) k_ut_init_b(long long R, const Seg *seg, long long *q, long long *a, long long *am) {
    FOR_EACH(i, R) {
        const long long pr = seg[i].prev;
        q[i] = pr < 0 ? i : pr;
        a[i] = pr < 0 ? 0 : seg[pr].len;
        am[i] = pr < 0 ? 0 : seg[pr].mult;
    }
}

// a[i] = edges of the rulers in [q[i], i) along the list; a root points to itself with a = 0
__global__ void __launch_bounds__(TPB, 4) k_ut_jump_b(long long R, const long long *q, const long long *a, const long long *am,
                                                   long long *q2, long long *a2, long long *am2) {
    FOR_EACH(i, R) {
        const long long h = q[i];
        q2[i] = q[h];
        a2[i] = a[i] + a[h];
        am2[i] = am[i] + am[h];
    }
}

__global__ void __launch_bounds__(TPB) k_ut_tot(long long R, Seg *seg, const long long *q, const long long *a, const long long *am) {
    FOR_EACH(i, R) {
        const long long nx = seg[i].next;
        if (nx < 0 || seg[nx].prev < 0) {                            // the tail of its list
            Seg &h = seg[q[i]];
            h.tot_len = a[i] + seg[i].len;
            h.tot_mult = am[i] + seg[i].mult;
        }
    }
}

// rof -> e1 of the edge's unitig, off -> offset in it; the last edge records itself under e1
__global__ void __launch_bounds__(TPB) k_ut_place(long long n, const Seg *seg, const long long *q, const long long *a, long long *rof,
                                                  long long *off, long long *last) {
    FOR_EACH(x, n) {
        const long long i = rof[x];
        if (i < 0) continue;
        const Seg &h = seg[q[i]];
        const long long len = h.tot_len;
        long long pos = a[i] + off[x], e1 = h.edge;
        if (h.flags & 1) { e1 = h.mn; pos = (pos - h.mnoff + len) % len; }
        rof[x] = e1;
        off[x] = pos;
        if (pos == len - 1) last[e1] = x;
    }
}

__global__ void __launch_bounds__(TPB, 4) k_ut_table(const QueryParams P, long long R, Seg *seg, const long long *head, const long long *last,
                                                  long long *keep) {
    FOR_EACH(i, R) if (seg[i].prev < 0) {
        Seg &s = seg[i];
        const long long e1 = (s.flags & 1) ? s.mn : s.edge;
        const long long rc = revcomp(P, last[e1]);
        const long long pe = rc >= 0 ? head[rc] : e1;
        const bool kept = e1 <= pe;
        s.flags |= (pe == e1 && rc >= 0 ? 2 : 0) | (kept ? 4 : 0);
        keep[e1] = kept;
    }
}

__global__ void __launch_bounds__(TPB) k_ut_rows(long long R, const Seg *seg, const long long *keep, const long long *last, int k,
                                                 int need_mult, long long *rows, long long *chars) {
    FOR_EACH(i, R) if (seg[i].prev < 0 && (seg[i].flags & 4)) {
        const Seg &s = seg[i];
        const long long e1 = (s.flags & 1) ? s.mn : s.edge;
        long long *r = rows + keep[e1] * 6;
        r[0] = e1; r[1] = last[e1]; r[2] = s.tot_len; r[4] = need_mult ? s.tot_mult : -1; r[5] = s.flags & 3;
        chars[keep[e1]] = k + s.tot_len;
    }
}

__global__ void __launch_bounds__(TPB) k_ut_seq_offset(long long U, const long long *chars, long long *rows) {
    FOR_EACH(r, U) rows[r * 6 + 3] = chars[r];
}

__global__ void __launch_bounds__(TPB) k_ut_scatter(const QueryParams P, const long long *head, const long long *off, const long long *keep,
                                                    const long long *rows, char *seq) {
    FOR_EACH(x, P.size) {
        const long long e1 = head[x];
        if (e1 < 0 || keep[e1 + 1] == keep[e1]) continue;
        char *s = seq + rows[keep[e1] * 6 + 3];
        const long long pos = off[x];
        s[P.k + pos] = "ACGT"[(get_w(P, x) - 1) & 3];
        if (pos == 0) {
            uint32_t lab[MAX_WPT];
            label(P, x, lab);
            for (int j = 0; j < P.k; ++j) s[j] = "ACGT"[kmer_char(lab, j)];
        }
    }
}

// frees the scratch buffers on every return path
struct Scratch {
    mgta_sdbg *g;
    ~Scratch() {
        for (DevBuf *b : {&g->ut_edge, &g->ut_seg, &g->ut_jump}) { cudaFree(b->p); b->p = nullptr; b->cap = 0; }
    }
};

int read_ll(mgta_sdbg *g, const long long *d, long long *out) {
    SCK(cudaMemcpyAsync(out, d, 8, cudaMemcpyDeviceToHost, g->stream));
    SCK(cudaStreamSynchronize(g->stream));
    return MGTA_OK;
}

size_t up256(size_t b) { return (b + 255) & ~(size_t)255; }

int unitigs(mgta_sdbg *g) {
    QueryParams P;
    int rc;
    if ((rc = query_params(g, &P))) return rc;
    const long long E = g->n_edges;
    // MGTA_UT_STRIDE: one ruler per S edges of a unitig, besides its head (a test hook: 1 = every edge, huge = heads only)
    const long long S = std::max(1ll, env_ll("MGTA_UT_STRIDE", 128));
    Scratch guard{g};
    // per edge: succ (later the last edge of each unitig, under e1), rof (ruler, later e1), off, ruler ids / keep
    // flags (E + 1), has_pred; the tile sums of the scans; two counters
    const size_t ll = up256(8 * (size_t)E + 8), nt = (size_t)(E + SCAN_TILE - 1) / SCAN_TILE + 1;
    if ((rc = grow(g, g->ut_edge, 4 * ll + up256(E) + up256(8 * nt) + 256, 0))) return rc;
    char *base = (char *)g->ut_edge.p;
    long long *succ = (long long *)base, *rof = (long long *)(base + ll), *off = (long long *)(base + 2 * ll), *rid = (long long *)(base + 3 * ll);
    uint8_t *has_pred = (uint8_t *)(base + 4 * ll);
    long long *tile_sum = (long long *)(base + 4 * ll + up256(E));
    unsigned long long *counter = (unsigned long long *)(base + 4 * ll + up256(E) + up256(8 * nt));
    long long *last = succ;

    SCK(cudaMemsetAsync(has_pred, 0, (size_t)E, g->stream));
    SCK(cudaMemsetAsync(counter, 0, 8, g->stream));
    const unsigned ge = grid_for(E);
    k_ut_links<<<ge, TPB, 0, g->stream>>>(P, succ, rof, has_pred);
    k_ut_mark<<<ge, TPB, 0, g->stream>>>(E, succ, has_pred, S, rid);
    if ((rc = scan(g, rid, E, tile_sum))) return rc;
    long long R0 = 0, R = 0;
    if ((rc = read_ll(g, rid + E, &R0))) return rc;
    if ((rc = grow(g, g->ut_seg, sizeof(Seg) * std::max(1ll, R0), 0))) return rc;
    Seg *seg = (Seg *)g->ut_seg.p;
    k_ut_rulers<<<ge, TPB, 0, g->stream>>>(E, rid, seg, rof);
    k_ut_walk<<<grid_for(R0), TPB, 0, g->stream>>>(P, g->need_mult, succ, rof, off, seg, 0, R0);
    k_ut_count_unvisited<<<ge, TPB, 0, g->stream>>>(E, succ, rof, counter);
    SCK(cudaGetLastError());
    long long unvisited = 0;
    if ((rc = read_ll(g, (const long long *)counter, &unvisited))) return rc;
    R = R0;
    if (unvisited) {                                               // cycles without a ruler
        if ((rc = grow(g, g->ut_seg, sizeof(Seg) * (R0 + unvisited), sizeof(Seg) * R0))) return rc;
        seg = (Seg *)g->ut_seg.p;
        SCK(cudaMemcpyAsync(counter, &R0, 8, cudaMemcpyHostToDevice, g->stream));
        k_ut_resid<<<ge, TPB, 0, g->stream>>>(E, succ, rof, seg, counter);
        SCK(cudaGetLastError());
        if ((rc = read_ll(g, (const long long *)counter, &R))) return rc;
        k_ut_walk<<<grid_for(R - R0), TPB, 0, g->stream>>>(P, g->need_mult, succ, rof, off, seg, R0, R);
    }
    k_ut_prev<<<grid_for(R), TPB, 0, g->stream>>>(R, seg);

    // ruler list ranking: six arrays of R + 1 (the first is later the scan of the rows' lengths)
    const size_t rl = up256(8 * (size_t)(R + 1));
    if ((rc = grow(g, g->ut_jump, 6 * rl, 0))) return rc;
    long long *J[6];
    for (int j = 0; j < 6; ++j) J[j] = (long long *)((char *)g->ut_jump.p + j * rl);
    int rounds = 0;
    while ((1ll << rounds) < R) ++rounds;
    const unsigned gr = grid_for(R);
    k_ut_init_a<<<gr, TPB, 0, g->stream>>>(R, seg, J[0], J[1]);
    for (int t = 0; t < rounds; ++t) {
        const int s = (t & 1) * 2, d = 2 - s;
        k_ut_jump_a<<<gr, TPB, 0, g->stream>>>(R, J[s], J[s + 1], J[d], J[d + 1]);
    }
    const int fa = (rounds & 1) * 2;
    k_ut_break<<<gr, TPB, 0, g->stream>>>(R, seg, J[fa], J[fa + 1]);
    k_ut_init_b<<<gr, TPB, 0, g->stream>>>(R, seg, J[0], J[1], J[2]);
    for (int t = 0; t < rounds; ++t) {
        const int s = (t & 1) * 3, d = 3 - s;
        k_ut_jump_b<<<gr, TPB, 0, g->stream>>>(R, J[s], J[s + 1], J[s + 2], J[d], J[d + 1], J[d + 2]);
    }
    const int fb = (rounds & 1) * 3;
    k_ut_tot<<<gr, TPB, 0, g->stream>>>(R, seg, J[fb], J[fb + 1], J[fb + 2]);
    k_ut_place<<<ge, TPB, 0, g->stream>>>(E, seg, J[fb], J[fb + 1], rof, off, last);

    // table: the kept unitigs in edge order
    long long *keep = rid;
    SCK(cudaMemsetAsync(keep, 0, 8 * (size_t)(E + 1), g->stream));
    k_ut_table<<<gr, TPB, 0, g->stream>>>(P, R, seg, rof, last, keep);
    if ((rc = scan(g, keep, E, tile_sum))) return rc;
    long long U = 0;
    if ((rc = read_ll(g, keep + E, &U))) return rc;
    if ((rc = grow(g, g->ut_rows, 48 * (size_t)std::max(1ll, U), 0))) return rc;
    long long *rows = (long long *)g->ut_rows.p, *chars = J[0];
    k_ut_rows<<<gr, TPB, 0, g->stream>>>(R, seg, keep, last, P.k, g->need_mult, rows, chars);
    if ((rc = scan(g, chars, U, tile_sum))) return rc;
    k_ut_seq_offset<<<grid_for(U), TPB, 0, g->stream>>>(U, chars, rows);
    long long n_chars = 0;
    if ((rc = read_ll(g, chars + U, &n_chars))) return rc;
    if ((rc = grow(g, g->ut_seq, (size_t)std::max(1ll, n_chars), 0))) return rc;
    k_ut_scatter<<<ge, TPB, 0, g->stream>>>(P, rof, off, keep, rows, (char *)g->ut_seq.p);
    SCK(cudaGetLastError());
    SCK(cudaStreamSynchronize(g->stream));
    g->ut_n_rows = U;
    g->ut_n_chars = (unsigned long long)n_chars;
    return MGTA_OK;
}

// ---- links between the unitigs ------------------------------------------------------------------------------------------
__device__ __forceinline__ long long ul_bar(const long long *rows, long long o) { return (rows[(o >> 1) * 6 + 5] & 2) ? o : o ^ 1; }

__global__ void __launch_bounds__(TPB, 4) k_ul_heads(const QueryParams P, long long U, const long long *rows, long long *hid,
                                                  long long *end1) {
    FOR_EACH(i, 2 * U) {
        const long long r = i >> 1, *w = rows + r * 6;
        const bool side = i & 1;
        if (w[5] & 1) continue;                                    // a cycle has no head
        if (!side) hid[w[0]] = 2 * r;
        if (w[5] & 2) continue;
        // one call site for both sides: a warp whose lanes took two calls would run them one after the other
        const long long x = revcomp(P, w[side ? 0 : 1]);
        if (side) end1[r] = x;
        else if (x >= 0) hid[x] = 2 * r + 1;                       // x = -1 only for an invalid edge: never a row's last
    }
}

// the canonical links out of oriented unitig o: their `to` values ascending in to[] -> their number (at most 4)
__device__ __forceinline__ int ul_links_of(const QueryParams &P, const long long *rows, const long long *hid, const long long *end1,
                                           long long o, long long *to) {
    const long long r = o >> 1, fl = rows[r * 6 + 5];
    if (fl & 1) {                                                  // a cycle: (2r, 2r) only
        to[0] = o;
        return (o & 1) ? 0 : 1;
    }
    if ((o & 1) && (fl & 2)) return 0;                             // a SELF_RC row has no 2r + 1
    long long out[4];
    const int n = outgoing(P, forward(P, (o & 1) ? end1[r] : rows[r * 6 + 1]), out);
    const long long ba = ul_bar(rows, o);
    int c = 0;
    for (int j = 0; j < n; ++j) {
        const long long b = hid[out[j]], bb = ul_bar(rows, b);
        if (o < bb || (o == bb && b <= ba)) {                      // (o, b) <= (bar(b), bar(o))
            int p = c++;
            for (; p > 0 && to[p - 1] > b; --p) to[p] = to[p - 1];
            to[p] = b;
        }
    }
    return c;
}

__global__ void __launch_bounds__(TPB) k_ul_count(const QueryParams P, long long n_or, const long long *rows, const long long *hid,
                                                  const long long *end1, long long *cnt) {
    FOR_EACH(o, n_or) {
        long long to[4];
        cnt[o] = ul_links_of(P, rows, hid, end1, o, to);
    }
}

__global__ void __launch_bounds__(TPB) k_ul_write(const QueryParams P, long long n_or, const long long *rows, const long long *hid,
                                                  const long long *end1, const long long *off, long long *links) {
    FOR_EACH(o, n_or) {
        long long to[4];
        const int n = ul_links_of(P, rows, hid, end1, o, to);
        for (int j = 0; j < n; ++j) {
            links[(off[o] + j) * 2] = o;
            links[(off[o] + j) * 2 + 1] = to[j];
        }
    }
}

int unitig_links(mgta_sdbg *g) {
    QueryParams P;
    int rc;
    if ((rc = query_params(g, &P))) return rc;
    const long long E = g->n_edges, U = g->ut_n_rows, NO = 2 * U;
    Scratch guard{g};
    // hid per edge, end(2r + 1) per row, link counts per oriented unitig (NO + 1: the scan's total), the scan's tile sums
    const size_t he = up256(8 * (size_t)E), hr = up256(8 * (size_t)U), ho = up256(8 * (size_t)(NO + 1));
    const size_t nt = (size_t)(NO + SCAN_TILE - 1) / SCAN_TILE + 1;
    if ((rc = grow(g, g->ut_edge, he + hr + ho + up256(8 * nt), 0))) return rc;
    char *base = (char *)g->ut_edge.p;
    long long *hid = (long long *)base, *end1 = (long long *)(base + he), *cnt = (long long *)(base + he + hr);
    long long *tile_sum = (long long *)(base + he + hr + ho);
    const long long *rows = (const long long *)g->ut_rows.p;
    const unsigned go = grid_for(NO);
    k_ul_heads<<<go, TPB, 0, g->stream>>>(P, U, rows, hid, end1);
    k_ul_count<<<go, TPB, 0, g->stream>>>(P, NO, rows, hid, end1, cnt);
    if ((rc = scan(g, cnt, NO, tile_sum))) return rc;
    long long L = 0;
    if ((rc = read_ll(g, cnt + NO, &L))) return rc;
    if ((rc = grow(g, g->ul_links, 16 * (size_t)std::max(1ll, L), 0))) return rc;
    k_ul_write<<<go, TPB, 0, g->stream>>>(P, NO, rows, hid, end1, cnt, (long long *)g->ul_links.p);
    SCK(cudaGetLastError());
    SCK(cudaStreamSynchronize(g->stream));
    g->ul_n_links = L;
    return MGTA_OK;
}

}  // namespace

extern "C" int mgta_sdbg_unitigs(mgta_sdbg *g, int64_t *n_rows, uint64_t *n_chars) {
    if (!g) return MGTA_ERR_ARG;
    if (!n_rows || !n_chars) { g->err = "sdbg_unitigs: null n_rows / n_chars"; return MGTA_ERR_ARG; }
    if (!g->finished) { g->err = "sdbg_unitigs: call mgta_sdbg_finish first"; return MGTA_ERR_STATE; }
    SCK(cudaSetDevice(g->device));
    g->ut_ready = false;
    g->ul_ready = false;                                           // the links name rows of the previous call
    int rc;
    if ((rc = unitigs(g))) return rc;
    g->ut_ready = true;
    *n_rows = g->ut_n_rows;
    *n_chars = g->ut_n_chars;
    return MGTA_OK;
}

extern "C" int mgta_sdbg_unitig_copy(mgta_sdbg *g, void *rows, uint64_t rows_bytes, void *seq, uint64_t seq_bytes) {
    if (!g) return MGTA_ERR_ARG;
    if (!g->ut_ready) { g->err = "sdbg_unitig_copy: call mgta_sdbg_unitigs first"; return MGTA_ERR_STATE; }
    const uint64_t need_rows = 48ull * (uint64_t)g->ut_n_rows, need_seq = g->ut_n_chars;
    char b[160];
    if (need_rows && (!rows || rows_bytes < need_rows)) {
        snprintf(b, sizeof(b), "sdbg_unitig_copy: rows buffer of %llu bytes, %llu needed", (unsigned long long)rows_bytes, (unsigned long long)need_rows);
        g->err = b;
        return MGTA_ERR_ARG;
    }
    if (need_seq && (!seq || seq_bytes < need_seq)) {
        snprintf(b, sizeof(b), "sdbg_unitig_copy: seq buffer of %llu bytes, %llu needed", (unsigned long long)seq_bytes, (unsigned long long)need_seq);
        g->err = b;
        return MGTA_ERR_ARG;
    }
    SCK(cudaSetDevice(g->device));
    if (need_rows)
        SCK(cudaMemcpyAsync(rows, g->ut_rows.p, need_rows, on_device(rows) ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, g->stream));
    if (need_seq)
        SCK(cudaMemcpyAsync(seq, g->ut_seq.p, need_seq, on_device(seq) ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, g->stream));
    SCK(cudaStreamSynchronize(g->stream));
    return MGTA_OK;
}

extern "C" int mgta_sdbg_unitig_links(mgta_sdbg *g, int64_t *n_links) {
    if (!g) return MGTA_ERR_ARG;
    if (!n_links) { g->err = "sdbg_unitig_links: null n_links"; return MGTA_ERR_ARG; }
    if (!g->ut_ready) { g->err = "sdbg_unitig_links: call mgta_sdbg_unitigs first"; return MGTA_ERR_STATE; }
    SCK(cudaSetDevice(g->device));
    g->ul_ready = false;
    int rc;
    if ((rc = unitig_links(g))) return rc;
    g->ul_ready = true;
    *n_links = g->ul_n_links;
    return MGTA_OK;
}

extern "C" int mgta_sdbg_unitig_link_copy(mgta_sdbg *g, void *links, uint64_t bytes) {
    if (!g) return MGTA_ERR_ARG;
    if (!g->ul_ready) { g->err = "sdbg_unitig_link_copy: call mgta_sdbg_unitig_links after mgta_sdbg_unitigs first"; return MGTA_ERR_STATE; }
    const uint64_t need = 16ull * (uint64_t)g->ul_n_links;
    if (need && (!links || bytes < need)) {
        char b[160];
        snprintf(b, sizeof(b), "sdbg_unitig_link_copy: links buffer of %llu bytes, %llu needed", (unsigned long long)bytes, (unsigned long long)need);
        g->err = b;
        return MGTA_ERR_ARG;
    }
    SCK(cudaSetDevice(g->device));
    if (need)
        SCK(cudaMemcpyAsync(links, g->ul_links.p, need, on_device(links) ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, g->stream));
    SCK(cudaStreamSynchronize(g->stream));
    return MGTA_OK;
}
