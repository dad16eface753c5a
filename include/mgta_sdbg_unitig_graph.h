/* mgta_sdbg_unitig_graph.h -- the unitig graph of a device SdBG: which unitig continues into which, as oriented links
 * between the rows of mgta_sdbg_unitigs (include/mgta_sdbg_unitig.h), computed in HBM.
 *
 * Terms of include/mgta_sdbg_unitig.h: valid edge, succ, unitig, kept row, the CYCLE (1) / SELF_RC (2) flags, rows sorted
 * by first_edge.  A linear row is one without the CYCLE flag.
 *
 *   oriented unitig  o = 2r + s for row r: s = 0 is the row's sequence, s = 1 its reverse complement (the discarded
 *                    partner unitig).  A SELF_RC row has only o = 2r.
 *   bar(o)           the reverse orientation: o ^ 1, except bar(2r) = 2r for a SELF_RC row.
 *   end(o)           for a linear o: end(2r) = last_edge(r), end(2r + 1) = REVCOMP(first_edge(r)) (the partner's last edge).
 *   id(f)            for an edge f that starts a linear unitig: 2r when f = first_edge(r), else 2r + 1 for the row r whose
 *                    last_edge is REVCOMP(f).  Exactly one holds: REVCOMP is -1 only for invalid edges.
 *   links F          for every linear oriented unitig a with t = FORWARD(end(a)): (a, id(f)) for every valid out-edge f of t
 *                    (OUTGOING(t); t does not have in-degree 1 and out-degree 1, so every such f starts a linear unitig);
 *                    and (2r, 2r) for every cycle row (a cycle's sequence ends on the k characters it starts with).  F is
 *                    closed under the twin map (a, b) -> (bar(b), bar(a)) and has no duplicates.
 *   output           the canonical links: the pairs (a, b) of F with (a, b) <= (bar(b), bar(a)) (lexicographic), as
 *                    int64 x 2 rows (from, to) sorted by (from, to); each twin pair appears once, as in GFA.
 * Equivalently a -> b exactly when the last k characters of a's sequence equal the first k of b's, k the node length
 * (a unitig of n edges has k + n characters).  The overlap of every link is k.
 */
#ifndef MGTA_SDBG_UNITIG_GRAPH_H
#define MGTA_SDBG_UNITIG_GRAPH_H

#include "mgta_cuda.h"

#ifdef __cplusplus
extern "C" {
#endif

/* computes the canonical links between the rows of the last mgta_sdbg_unitigs on the graph's stream and returns when
 * their number *n_links is known.  The links stay in a device buffer owned by the graph until the next call or
 * mgta_sdbg_destroy; the rows and sequence of mgta_sdbg_unitigs do not change.  MGTA_ERR_STATE before mgta_sdbg_unitigs. */
int mgta_sdbg_unitig_links(mgta_sdbg *g, int64_t *n_links);

/* copies the links of the last mgta_sdbg_unitig_links: n_links * 16 bytes, to host or device memory.  MGTA_ERR_ARG when
 * the buffer is too small (the message names it), MGTA_ERR_STATE when no links were computed since the last
 * mgta_sdbg_unitigs (their row numbers would refer to older rows).  The graph, its queries, its unitigs and its links stay
 * usable after every error. */
int mgta_sdbg_unitig_link_copy(mgta_sdbg *g, void *links, uint64_t bytes);

#ifdef __cplusplus
}
#endif

#endif
