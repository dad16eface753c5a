// sdbg_query.cu -- batched navigation queries on the device SdBG (include/mgta_sdbg_query.h): the SuccinctDBG member
// functions IndexBinarySearch, Label, Forward, Backward, Outdegree / Indegree, OutgoingEdges / IncomingEdges,
// EdgeMultiplicity and EdgeReverseComplement, as BOSS rank / select chains over the tables sdbg_index.cu built.
// One thread per query row; the navigation itself (rank / select, node ranges, LOOKUP) lives in sdbg_nav.cuh.
#include <string.h>

#include "sdbg_nav.cuh"
#include "../../include/mgta_sdbg_query.h"

using namespace mgta_sdbg_impl;

namespace {

template <int OP>
__global__ void __launch_bounds__(256) k_sdbg_query(const QueryParams P) {
    for (unsigned long long q = blockIdx.x * 256ull + threadIdx.x; q < P.n; q += (unsigned long long)gridDim.x * 256ull) {
        if (OP == MGTA_SQ_LOOKUP) {
            uint32_t x[MAX_WPT];
            const uint32_t *in = (const uint32_t *)P.in + q * P.wpt;
            for (int j = 0; j < P.wpt; ++j) x[j] = in[j];
            ((long long *)P.out)[q] = lookup(P, x);
            continue;
        }
        const long long i = ((const long long *)P.in)[q];
        const bool ok = i >= 0 && i < P.size;
        if (!ok) atomicMin(P.bad_row, P.row0 + q);
        if (OP == MGTA_SQ_LABEL) {
            uint32_t x[MAX_WPT];
            uint32_t *out = (uint32_t *)P.out + q * (P.wpt + 1);
            const int t = ok ? label(P, i, x) : 0;
            for (int j = 0; j < P.wpt; ++j) out[j] = ok ? x[j] : 0u;
            out[P.wpt] = (uint32_t)t;
        } else if (OP == MGTA_SQ_OUTGOING || OP == MGTA_SQ_INCOMING) {
            long long e[4] = {-1, -1, -1, -1};
            if (ok) { if (OP == MGTA_SQ_OUTGOING) outgoing(P, i, e); else incoming(P, i, e); }
            long long *out = (long long *)P.out + q * 4;
            for (int j = 0; j < 4; ++j) out[j] = e[j];
        } else {
            long long r = -1;
            if (ok) {
                long long e[4];
                if (OP == MGTA_SQ_FORWARD) r = forward(P, i);
                if (OP == MGTA_SQ_BACKWARD) r = backward(P, i);
                if (OP == MGTA_SQ_OUTDEGREE) r = outgoing(P, i, e);
                if (OP == MGTA_SQ_INDEGREE) r = incoming(P, i, e);
                if (OP == MGTA_SQ_MULTIPLICITY) r = multiplicity(P, i);
                if (OP == MGTA_SQ_REVCOMP) r = revcomp(P, i);
            }
            ((long long *)P.out)[q] = r;
        }
    }
}

bool row_bytes(int wpt, int op, uint64_t *in_row, uint64_t *out_row) {
    if (op < MGTA_SQ_LOOKUP || op > MGTA_SQ_REVCOMP) return false;
    *in_row = op == MGTA_SQ_LOOKUP ? 4ull * wpt : 8ull;
    *out_row = op == MGTA_SQ_LABEL ? 4ull * (wpt + 1) : (op == MGTA_SQ_OUTGOING || op == MGTA_SQ_INCOMING ? 32ull : 8ull);
    return true;
}

int launch(mgta_sdbg *g, int op, const QueryParams &P) {
    const unsigned grid = (unsigned)std::max(1ull, std::min((P.n + 255) / 256, 148ull * 64));
    switch (op) {
#define SQ_CASE(o) case o: k_sdbg_query<o><<<grid, 256, 0, g->stream>>>(P); break;
        SQ_CASE(MGTA_SQ_LOOKUP) SQ_CASE(MGTA_SQ_LABEL) SQ_CASE(MGTA_SQ_FORWARD) SQ_CASE(MGTA_SQ_BACKWARD) SQ_CASE(MGTA_SQ_OUTDEGREE)
        SQ_CASE(MGTA_SQ_INDEGREE) SQ_CASE(MGTA_SQ_OUTGOING) SQ_CASE(MGTA_SQ_INCOMING) SQ_CASE(MGTA_SQ_MULTIPLICITY) SQ_CASE(MGTA_SQ_REVCOMP)
#undef SQ_CASE
    }
    SCK(cudaGetLastError());
    return MGTA_OK;
}

}  // namespace

extern "C" int mgta_sdbg_query_row_bytes(const mgta_sdbg *g, int op, uint64_t *in_row, uint64_t *out_row) {
    if (!g || !in_row || !out_row) return MGTA_ERR_ARG;
    return row_bytes(g->wpt, op, in_row, out_row) ? MGTA_OK : MGTA_ERR_ARG;
}

extern "C" int mgta_sdbg_query(mgta_sdbg *g, int op, const void *in, uint64_t n, void *out, uint64_t out_bytes) {
    if (!g) return MGTA_ERR_ARG;
    uint64_t in_row = 0, out_row = 0;
    if (!row_bytes(g->wpt, op, &in_row, &out_row)) { g->err = "sdbg_query: unknown op " + std::to_string(op); return MGTA_ERR_ARG; }
    if (!g->finished) { g->err = "sdbg_query: call mgta_sdbg_finish first"; return MGTA_ERR_STATE; }
    if (op == MGTA_SQ_MULTIPLICITY && !g->need_mult) { g->err = "sdbg_query: MULTIPLICITY needs a graph built with need_multiplicity"; return MGTA_ERR_STATE; }
    if (n == 0) return MGTA_OK;
    if (!in || !out) { g->err = "sdbg_query: null in / out"; return MGTA_ERR_ARG; }
    if (out_bytes / out_row < n) { g->err = "sdbg_query: out_bytes < n * out_row"; return MGTA_ERR_ARG; }
    SCK(cudaSetDevice(g->device));
    int rc;
    QueryParams P;
    if ((rc = query_params(g, &P))) return rc;
    if (!env_ll("MGTA_SQ_LV1", 1)) P.bucket_start = nullptr;      // A/B: LOOKUP without the lv1 start
    if ((rc = grow(g, g->q_err, 64, 0))) return rc;
    const bool in_dev = on_device(in), out_dev = on_device(out);
    // host rows go through device buffers of at most `chunk` rows (MGTA_SQ_CHUNK_ROWS: a test hook)
    const unsigned long long chunk = in_dev && out_dev ? n : (unsigned long long)std::max(1ll, env_ll("MGTA_SQ_CHUNK_ROWS", 1ll << 22));
    if (!in_dev && (rc = grow(g, g->q_in, std::min<unsigned long long>(chunk, n) * in_row, 0))) return rc;
    if (!out_dev && (rc = grow(g, g->q_out, std::min<unsigned long long>(chunk, n) * out_row, 0))) return rc;
    SCK(cudaMemsetAsync(g->q_err.p, 0xFF, 8, g->stream));
    P.bad_row = (unsigned long long *)g->q_err.p;
    for (unsigned long long row0 = 0; row0 < n; row0 += chunk) {
        const unsigned long long cnt = std::min<unsigned long long>(chunk, n - row0);
        const char *src = (const char *)in + row0 * in_row;
        char *dst = (char *)out + row0 * out_row;
        if (!in_dev) SCK(cudaMemcpyAsync(g->q_in.p, src, cnt * in_row, cudaMemcpyHostToDevice, g->stream));
        P.in = in_dev ? (const void *)src : g->q_in.p;
        P.out = out_dev ? (void *)dst : g->q_out.p;
        P.n = cnt; P.row0 = row0;
        if ((rc = launch(g, op, P))) return rc;
        if (!out_dev) SCK(cudaMemcpyAsync(dst, g->q_out.p, cnt * out_row, cudaMemcpyDeviceToHost, g->stream));
    }
    unsigned long long bad = 0;
    SCK(cudaMemcpyAsync(&bad, g->q_err.p, 8, cudaMemcpyDeviceToHost, g->stream));
    SCK(cudaStreamSynchronize(g->stream));
    if (bad != ~0ull) {
        long long id = 0;
        SCK(cudaMemcpyAsync(&id, (const char *)in + bad * 8, 8, cudaMemcpyDefault, g->stream));
        SCK(cudaStreamSynchronize(g->stream));
        char b[160];
        snprintf(b, sizeof(b), "sdbg_query: row %llu: edge id %lld outside [0, %lld)", bad, id, g->n_edges);
        g->err = b;
        return MGTA_ERR_ARG;
    }
    return MGTA_OK;
}
