/* mgta_sdbg_query.h -- batched navigation queries on a finished device SdBG (mgta_sdbg, include/mgta_cuda.h).
 *
 * One row in, one row out, one device thread per row.  Every query reads the arrays and rank / select tables that
 * mgta_sdbg_finish left in HBM; nothing is copied to the host.
 *
 * Notation: order k; edge i in [0, size) belongs to node v(i) (k characters) and carries W(i): 0 = '$', 1..4 = ACGT,
 * 5..8 = the same characters flagged (an earlier node already has an edge into the same target).  A tip node is a dummy
 * node whose label starts with '$'; its edges have is_tip set.  valid = !(is_tip | W == 0).
 *
 * Row formats (wpt = words_per_tip_label = ceil(2k / 32)):
 *   k-mer    wpt u32, forward orientation, first character in bits 31..30 of word 0, A C G T = 0..3, unused low bits 0
 *   edge id  i64; -1 means "none"
 *
 *   op            in row    out row
 *   LOOKUP        k-mer     i64: the last edge (last = 1) of node X, or -1 (tip nodes are never found)
 *   LABEL         edge id   k-mer of v(i) + u32 (1 when v(i) is a tip node; its '$' is packed as 0)
 *   FORWARD       edge id   i64: last edge of the target node; -1 for W = 0
 *   BACKWARD      edge id   i64: the edge with the unflagged W = last character of v(i) entering v(i); -1 for a tip node
 *   OUTDEGREE     edge id   i64: valid edges leaving v(i) (0 for a tip node)
 *   INDEGREE      edge id   i64: valid edges entering v(i) (0 for a tip node)
 *   OUTGOING      edge id   4 x i64: the valid edges leaving v(i) in edge order, padded with -1
 *   INCOMING      edge id   4 x i64: the valid edges entering v(i) in edge order, padded with -1
 *   MULTIPLICITY  edge id   i64: edge_multi, or the large list's value when edge_multi is 255
 *   REVCOMP       edge id   i64: the edge whose (k+1)-mer label.W is the reverse complement of edge i's; -1 if i is invalid
 */
#ifndef MGTA_SDBG_QUERY_H
#define MGTA_SDBG_QUERY_H

#include "mgta_cuda.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    MGTA_SQ_LOOKUP = 1,
    MGTA_SQ_LABEL,
    MGTA_SQ_FORWARD,
    MGTA_SQ_BACKWARD,
    MGTA_SQ_OUTDEGREE,
    MGTA_SQ_INDEGREE,
    MGTA_SQ_OUTGOING,
    MGTA_SQ_INCOMING,
    MGTA_SQ_MULTIPLICITY,
    MGTA_SQ_REVCOMP
} mgta_sdbg_query_op;

/* bytes of one input and one output row of `op` on graph g (g may be unfinished: the row sizes depend on k only) */
int mgta_sdbg_query_row_bytes(const mgta_sdbg *g, int op, uint64_t *in_row, uint64_t *out_row);

/* runs `op` on n rows.  `in` and `out` may each be host or device memory; host input is staged through bounded device
 * buffers, so n may exceed free HBM.  Runs on the graph's stream and returns when `out` holds every result.
 * MGTA_ERR_STATE: before mgta_sdbg_finish, or MULTIPLICITY on a graph created with need_multiplicity = 0.
 * MGTA_ERR_ARG: unknown op, out_bytes < n * out_row, or an edge id outside [0, size) (the message names the first bad row).
 * The graph stays usable after every error. */
int mgta_sdbg_query(mgta_sdbg *g, int op, const void *in, uint64_t n, void *out, uint64_t out_bytes);

#ifdef __cplusplus
}
#endif

#endif
