/* mgta_sdbg_unitig.h -- the unitigs (maximal non-branching paths) of a finished device SdBG (mgta_sdbg, include/mgta_cuda.h),
 * spelled out as sequence, computed in HBM.
 *
 * Conventions of include/mgta_sdbg_query.h: an edge is valid when !(is_tip | W == 0); OUTDEGREE and INDEGREE count
 * valid edges only.
 *
 *   succ(e)   for a valid edge e with target node t = FORWARD(e): the single valid out-edge of t when outdeg(t) == 1 and
 *             indeg(t) == 1, else none.  Every valid edge has at most one predecessor.
 *   unitig    a maximal chain e1 -> ... -> en under succ; every valid edge lies in exactly one.  A linear unitig starts
 *             at a valid edge without predecessor; in a cycle every edge has one, and e1 is its smallest edge id.
 *   sequence  LABEL(v(e1)) (k characters), then W(e1) ... W(en): k + n characters of ASCII ACGT.  A cycle is spelled the
 *             same way, so its last k characters repeat its first k.
 *   pairing   the reverse complement of unitig U is the unitig holding REVCOMP(en) (for a linear unitig that edge is the
 *             partner's e1).  U is kept when e1(U) <= e1(that unitig), so one unitig of every pair is kept; a unitig
 *             that is its own reverse complement is kept once and flagged.
 *
 * Rows (int64 x 6, sorted by first_edge):  first_edge, last_edge, n_edges, seq_offset, mult_sum, flags
 *   mult_sum  sum of the edge multiplicities (MULTIPLICITY), or -1 on a graph created with need_multiplicity = 0
 *   flags     1 = cycle, 2 = its own reverse complement
 * Sequence buffer: the kept sequences concatenated in row order; seq_offset is a row's start in it.
 * Check: the sum over rows of n_edges * (flags & 2 ? 1 : 2) equals the number of valid edges.
 */
#ifndef MGTA_SDBG_UNITIG_H
#define MGTA_SDBG_UNITIG_H

#include "mgta_cuda.h"

#ifdef __cplusplus
extern "C" {
#endif

/* computes the unitigs on the graph's stream and returns when their counts are known: *n_rows rows and *n_chars
 * characters of sequence.  The results stay in device buffers owned by the graph until the next call or
 * mgta_sdbg_destroy.  MGTA_ERR_STATE before mgta_sdbg_finish. */
int mgta_sdbg_unitigs(mgta_sdbg *g, int64_t *n_rows, uint64_t *n_chars);

/* copies the results of the last mgta_sdbg_unitigs: n_rows * 48 bytes of rows and n_chars bytes of sequence.  Either
 * destination may be host or device memory.  MGTA_ERR_ARG when a buffer is too small (the message names it),
 * MGTA_ERR_STATE before mgta_sdbg_unitigs.  The graph, its queries and its results stay usable after every error. */
int mgta_sdbg_unitig_copy(mgta_sdbg *g, void *rows, uint64_t rows_bytes, void *seq, uint64_t seq_bytes);

#ifdef __cplusplus
}
#endif

#endif
