// sdbg_index.cu -- SdBG load + rank/select build on the device (SURVEY 8f row 3).
//
// Replaces, for a record stream that is already in HBM (or is handed over from the host), the serial u16-at-a-time loop of
// SuccinctDBG::LoadFromMultiFile (reference succinct_dbg.cpp:595-723), SuccinctDBG::init (succinct_dbg.h:62-83) and the
// table builds RankAndSelect4Bits::Build (rank_and_select.h:81-150) / RankAndSelect1Bit::Build (rank_and_select.h:420-487).
// Every array has the reference's layout bit for bit (tests compare with a dump of the reference's own members):
//
//   w        4 bits per edge, 16 per u64, edge i at bits 4 (i % 16)        (succinct_dbg.cpp:655-662)
//   last, is_tip, invalid (= is_tip | W == 0), is_multi_1                  1 bit per edge, 64 per u64 (:664-686, init)
//   edge_multi u8 per edge (255 = look in the large list), large list (edge, multiplicity) in edge order (:680-704)
//   tip_node_seq  words_per_tip_label u32 per tip, in edge order           (:706-709)
//   rank tables   major (i64 every 65536) + minor (u16 every 256) exclusive counts, per W character / for last / is_tip
//   select tables rank_to_interval: the 256-interval holding every 256th occurrence
//   f, rank_f
//
// k_sdbg_parse: one warp per lv1 bucket walks the bucket's u16 words 32 at a time.  A window whose 32 words carry no tip
// and no large-multiplicity flag is 32 one-word records (the usual case); otherwise the record starts are the orbit of
// the first header under "skip my payload", walked with one shuffle per record.  The records of a window are compacted
// to the low lanes, and a window leaves as a handful of word-wide atomicOr (ballots for the bit vectors, an 8-lane
// butterfly for the W nibbles) instead of four atomics per record.
#include <string.h>

#include "sdbg_index.cuh"

using namespace mgta_sdbg_impl;

namespace {

constexpr int NB = 65536;
constexpr int PARSE_WARPS = 8;

struct ParseParams {
    const uint16_t *stream;            // records of buckets [b0, b1), bucket order
    const unsigned long long *base;    // [n][4]: u16 offset in stream, first edge, first tip, first large multiplicity
    const long long *meta;             // [n][3]: items, tips, large (device copy)
    int n_buckets, wpt;
    int need_mult;
    uint32_t *w, *last, *tip, *invalid, *multi1;
    uint8_t *edge_multi;
    uint32_t *tip_seq;
    unsigned long long *large_edge;
    uint16_t *large_val;
    unsigned *err;
};

__global__ void __launch_bounds__(PARSE_WARPS * 32) k_sdbg_parse(const ParseParams P) {
    const unsigned lane = threadIdx.x & 31, lt = (1u << lane) - 1u;
    const int warp = (blockIdx.x * PARSE_WARPS) + (threadIdx.x >> 5), n_warps = gridDim.x * PARSE_WARPS;
    for (int b = warp; b < P.n_buckets; b += n_warps) {
        const unsigned long long items = (unsigned long long)P.meta[3 * b], tips = (unsigned long long)P.meta[3 * b + 1],
                                 large = (unsigned long long)P.meta[3 * b + 2];
        if (items == 0) continue;
        const unsigned long long n_words = items + large + 2ull * P.wpt * tips;
        const uint16_t *p = P.stream + P.base[4 * b];
        const unsigned long long e0 = P.base[4 * b + 1], t0 = P.base[4 * b + 2], l0 = P.base[4 * b + 3];
        unsigned long long rec = 0, n_tip = 0, n_large = 0;
        unsigned s = 0;                                            // lane of the first header of the window
        for (unsigned long long pos = 0; pos < n_words; pos += 32) {
            const unsigned long long idx = pos + lane;
            const bool valid = idx < n_words;
            const unsigned v = valid ? p[idx] : 0u;
            const unsigned tipf = (v >> 5) & 1u, lg = (v >> 8) == 255u ? 1u : 0u;
            const unsigned len = 1u + lg + tipf * 2u * (unsigned)P.wpt;
            const unsigned vmask = __ballot_sync(0xFFFFFFFFu, valid);
            const unsigned fmask = __ballot_sync(0xFFFFFFFFu, valid && (tipf | lg));
            unsigned hdr, s_next;
            if (s == 0 && fmask == 0) {
                hdr = vmask; s_next = 0;
            } else {
                hdr = 0;
                unsigned q = s;
                while (q < 32 && ((vmask >> q) & 1u)) {            // warp-uniform walk over the record starts
                    hdr |= 1u << q;
                    q += __shfl_sync(0xFFFFFFFFu, len, q);
                }
                s_next = q >= 32 ? q - 32 : 0;
            }
            const unsigned n = __popc(hdr);
            const bool is_hdr = (hdr >> lane) & 1u;
            // payload of the records that start in this window (may lie in the next window: read from global memory)
            const unsigned tmask = __ballot_sync(0xFFFFFFFFu, is_hdr && tipf), lmask = __ballot_sync(0xFFFFFFFFu, is_hdr && lg);
            if (is_hdr && lg && P.need_mult) {
                const unsigned long long li = l0 + n_large + __popc(lmask & lt);
                const unsigned long long e = e0 + rec + __popc(hdr & lt);
                if (idx + 1 < n_words) { P.large_edge[li] = e; P.large_val[li] = p[idx + 1]; } else atomicOr(P.err, 1u);
            }
            if (is_hdr && tipf) {
                const unsigned long long ti = t0 + n_tip + __popc(tmask & lt);
                const unsigned long long q0 = idx + 1 + lg;
                if (q0 + 2ull * P.wpt <= n_words) {
                    for (int j = 0; j < P.wpt; ++j) P.tip_seq[ti * P.wpt + j] = (uint32_t)p[q0 + 2 * j] | ((uint32_t)p[q0 + 2 * j + 1] << 16);
                } else {
                    atomicOr(P.err, 2u);
                }
            }
            // compact the records to lanes [0, n): lane j takes the j-th header
            const int src = __fns(hdr, 0, (int)lane + 1);
            const unsigned x = __shfl_sync(0xFFFFFFFFu, v, src < 0 ? 0 : src);
            const bool act = lane < n;
            const unsigned wc = act ? (x & 15u) : 0u;
            const unsigned long long i0 = e0 + rec;                 // edge of compacted lane 0
            const unsigned sh = (unsigned)(i0 & 31ull);
            const unsigned long long wi = i0 >> 5;
            const unsigned b_last = __ballot_sync(0xFFFFFFFFu, act && ((x >> 4) & 1u));
            const unsigned b_tip = __ballot_sync(0xFFFFFFFFu, act && ((x >> 5) & 1u));
            const unsigned b_inv = __ballot_sync(0xFFFFFFFFu, act && (((x >> 5) & 1u) || wc == 0u));
            const unsigned b_m1 = __ballot_sync(0xFFFFFFFFu, act && (x >> 8) <= 1u);
            if (lane < 4) {
                uint32_t *arr = lane == 0 ? P.last : (lane == 1 ? P.tip : (lane == 2 ? P.invalid : P.multi1));
                const unsigned bits = lane == 0 ? b_last : (lane == 1 ? b_tip : (lane == 2 ? b_inv : b_m1));
                if (arr) {
                    if (bits << sh) atomicOr(arr + wi, bits << sh);
                    if (sh && (bits >> (32 - sh))) atomicOr(arr + wi + 1, bits >> (32 - sh));
                }
            }
            // W: 8 nibbles per u32; V[t] = nibbles of compacted lanes [8t, 8t + 8)
            unsigned y = wc << (4 * (lane & 7));
            y |= __shfl_xor_sync(0xFFFFFFFFu, y, 1);
            y |= __shfl_xor_sync(0xFFFFFFFFu, y, 2);
            y |= __shfl_xor_sync(0xFFFFFFFFu, y, 4);
            const unsigned lo = __shfl_sync(0xFFFFFFFFu, y, (lane & 3) * 8), hi = __shfl_sync(0xFFFFFFFFu, y, ((lane + 3) & 3) * 8);
            if (lane < 5) {
                const unsigned sh4 = 4u * (unsigned)(i0 & 7ull);
                const unsigned a = lane < 4 ? lo : 0u, c = lane > 0 ? hi : 0u;
                const unsigned out = (a << sh4) | (sh4 ? c >> (32 - sh4) : 0u);
                if (out) atomicOr(P.w + (i0 >> 3) + lane, out);
            }
            if (P.need_mult && act) P.edge_multi[i0 + lane] = (uint8_t)(x >> 8);
            rec += n; n_tip += __popc(tmask); n_large += __popc(lmask);
            s = s_next;
        }
        if (lane == 0 && (rec != items || n_tip != tips || n_large != large)) atomicOr(P.err, 4u);
    }
}

// ---- rank tables ---------------------------------------------------------------------------------------------------
// One block = one major interval (65536 positions = 256 minor intervals).  NC = 9 (W characters) or 1 (bit vector).
// minor[c][m * 256 + t] = count of c in positions [m * 65536, m * 65536 + 256 t); tot[c][m] = count in the major interval.
template <int NC>
__global__ void __launch_bounds__(256) k_rank_minor(const unsigned long long *__restrict__ text, long long length, long long n_minor,
                                                    uint16_t *minor, long long *tot, long long n_major) {
    __shared__ unsigned s_w[NC][8];
    const long long m = blockIdx.x;
    const unsigned t = threadIdx.x, lane = t & 31, warp = t >> 5;
    constexpr int PER_WORD = NC == 9 ? 16 : 64, WORDS = 256 / PER_WORD;
    const long long n_words = (length + PER_WORD - 1) / PER_WORD;
    const long long w0 = (m * 256 + t) * WORDS;
    unsigned cnt[NC];
#pragma unroll
    for (int c = 0; c < NC; ++c) cnt[c] = 0;
    for (int j = 0; j < WORDS; ++j) {
        if (w0 + j >= n_words) break;
        const unsigned long long x = text[w0 + j];
        if (NC == 9) {
            // the unused characters of the last word are zero and the reference counts them as character 0
            // (CountCharInWord_ sees whole words, rank_and_select.h:118-120): char_frequency[0] and the closing entries of
            // character 0 include that padding, and so do these
#pragma unroll
            for (int c = 0; c < NC; ++c) cnt[c] += (unsigned)count_char(x, c);
        } else {
            cnt[0] += (unsigned)__popcll(x);
        }
    }
#pragma unroll
    for (int c = 0; c < NC; ++c) {
        unsigned x = cnt[c];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned y = __shfl_up_sync(0xFFFFFFFFu, x, o);
            if (lane >= (unsigned)o) x += y;
        }
        if (lane == 31) s_w[c][warp] = x;
        cnt[c] = x - cnt[c];                                       // exclusive inside the warp
    }
    __syncthreads();
#pragma unroll
    for (int c = 0; c < NC; ++c) {
        unsigned add = 0, total = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) { if ((unsigned)w < warp) add += s_w[c][w]; total += s_w[c][w]; }
        const long long i = m * 256 + t;
        if (i < n_minor) minor[(long long)c * n_minor + i] = (uint16_t)(cnt[c] + add);
        if (t == 0) tot[(long long)c * n_major + m] = total;
    }
}

// exclusive scan of the major totals (one block per character); major[c][n_major - 1] ends up as the total count
__global__ void __launch_bounds__(1024) k_rank_major(long long *tot_to_major, long long n_major, long long *freq) {
    __shared__ long long s_w[32];
    __shared__ long long s_carry;
    long long *a = tot_to_major + (long long)blockIdx.x * n_major;
    const unsigned t = threadIdx.x, lane = t & 31, warp = t >> 5;
    if (t == 0) s_carry = 0;
    __syncthreads();
    for (long long base = 0; base < n_major; base += 1024) {
        const long long i = base + t;
        const long long v = i < n_major ? a[i] : 0;
        long long x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long y = __shfl_up_sync(0xFFFFFFFFu, x, o);
            if (lane >= (unsigned)o) x += y;
        }
        if (lane == 31) s_w[warp] = x;
        __syncthreads();
        long long add = 0, total = 0;
        for (unsigned w = 0; w < 32; ++w) { if (w < warp) add += s_w[w]; total += s_w[w]; }
        const long long carry = s_carry;
        if (i < n_major) a[i] = carry + add + x - v;
        __syncthreads();
        if (t == 0) s_carry = carry + total;
        __syncthreads();
    }
    if (t == 0) freq[blockIdx.x] = s_carry;
}

// the entries past the last full major interval: minor entries of intervals that start at or after `length` hold
// total - major (rank_and_select.h:122-126, :462-464); the natural exclusive counts give exactly that, except that the
// closing minor entry may belong to a major interval the data never reaches
__global__ void k_rank_close(uint16_t *minor, const long long *major, const long long *freq, long long n_minor, long long n_major, int nc) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < nc) {
        const long long i = n_minor - 1;
        minor[(long long)c * n_minor + i] = (uint16_t)(freq[c] - major[(long long)c * n_major + i / 256]);
    }
}

// select samples: table[s] = (first interval i with Occ(i) > 256 s) - 1; the closing entry = n_minor - 1
// (rank_and_select.h:131-147, :466-483).  Occ(i) = major[i / 256] + minor[i].
__global__ void __launch_bounds__(256) k_select_table(const uint16_t *__restrict__ minor, const long long *__restrict__ major, long long n_minor,
                                                      long long count, uint32_t *table, long long n_table) {
    const long long s = (long long)blockIdx.x * 256 + threadIdx.x;
    if (s >= n_table) return;
    if (s == n_table - 1) { table[s] = (uint32_t)(n_minor - 1); return; }
    const long long target = s * 256;
    long long lo = 0, hi = n_minor - 1;                            // first i with Occ(i) > target (exists: Occ(n_minor - 1) = count > target)
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (major[mid / 256] + (long long)minor[mid] > target) hi = mid; else lo = mid + 1;
    }
    table[s] = (uint32_t)(lo - 1);
}

// number of ones in bits [0, pos) of a bit vector, from its tables
__global__ void k_rank1_at(const unsigned long long *__restrict__ text, const uint16_t *__restrict__ minor, const long long *__restrict__ major,
                           long long length, long long total, const long long *pos_in, long long *out, int n) {
    const int i = threadIdx.x;
    if (i < n) out[i] = rank1(text, minor, major, length, total, pos_in[i]);
}

}  // namespace

extern "C" int mgta_sdbg_create(int device, void *stream, int kmer_k, int need_multiplicity, mgta_sdbg **out) {
    if (!out || kmer_k < 1 || kmer_k > MGTA_MAX_K) return MGTA_ERR_ARG;
    *out = nullptr;
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || device < 0 || device >= n_dev) return MGTA_ERR_CUDA;   // no CPU fallback
    mgta_sdbg *g = new mgta_sdbg();
    g->device = device; g->need_mult = need_multiplicity ? 1 : 0; g->kmer_k = kmer_k; g->wpt = (2 * kmer_k + 31) / 32;
    if (cudaSetDevice(device) != cudaSuccess) { delete g; return MGTA_ERR_CUDA; }
    if (stream) g->stream = (cudaStream_t)stream;
    else {
        if (cudaStreamCreateWithFlags(&g->stream, cudaStreamNonBlocking) != cudaSuccess) { delete g; return MGTA_ERR_CUDA; }
        g->own_stream = true;
    }
    if (cudaMalloc(&g->d_err, 4) != cudaSuccess || cudaMemsetAsync(g->d_err, 0, 4, g->stream) != cudaSuccess) { delete g; return MGTA_ERR_CUDA; }
    *out = g;
    return MGTA_OK;
}

extern "C" void mgta_sdbg_destroy(mgta_sdbg *g) {
    if (!g) return;
    cudaSetDevice(g->device);
    cudaStreamSynchronize(g->stream);
    DevBuf *all[] = {&g->w, &g->last, &g->tip, &g->invalid, &g->multi1, &g->edge_multi, &g->tip_seq, &g->large_edge, &g->large_val,
                     &g->staging, &g->base, &g->meta, &g->w_minor, &g->w_major, &g->last_minor, &g->last_major, &g->tip_minor,
                     &g->tip_major, &g->last_sel, &g->small, &g->q_bucket, &g->q_in, &g->q_out, &g->q_err,
                     &g->ut_rows, &g->ut_seq, &g->ut_edge, &g->ut_seg, &g->ut_jump};
    for (DevBuf *b : all) cudaFree(b->p);
    for (auto &b : g->w_sel) cudaFree(b.p);
    cudaFree(g->d_err);
    if (g->own_stream) cudaStreamDestroy(g->stream);
    delete g;
}

extern "C" const char *mgta_sdbg_last_error(const mgta_sdbg *g) { return g ? g->err.c_str() : "null sdbg"; }

// records of buckets [b0, b1) in bucket order; `bytes` may be a host or a device pointer; `meta` is a host pointer
extern "C" int mgta_sdbg_append(mgta_sdbg *g, int32_t b0, int32_t b1, const void *bytes, uint64_t n_bytes, const int64_t *meta) {
    if (!g) return MGTA_ERR_ARG;
    if (g->finished) { g->err = "sdbg_append after sdbg_finish"; return MGTA_ERR_STATE; }
    if (b0 != g->next_bucket || b1 < b0 || b1 > NB || !meta) { g->err = "sdbg_append: deliveries must cover the buckets in ascending order"; return MGTA_ERR_ARG; }
    SCK(cudaSetDevice(g->device));
    const int n = b1 - b0;
    g->next_bucket = b1;
    if (n == 0) return MGTA_OK;
    std::vector<unsigned long long> base((size_t)n * 4);
    unsigned long long off16 = 0;
    long long e = g->n_edges, t = g->n_tips, l = g->n_large;
    for (int i = 0; i < n; ++i) {
        const long long items = meta[3 * i], tips = meta[3 * i + 1], large = meta[3 * i + 2];
        if (items < 0 || tips < 0 || large < 0 || tips > items || large > items) { g->err = "sdbg_append: bad bucket table"; return MGTA_ERR_ARG; }
        g->bucket_start[b0 + i] = e;
        base[4 * i] = off16; base[4 * i + 1] = (unsigned long long)e; base[4 * i + 2] = (unsigned long long)t; base[4 * i + 3] = (unsigned long long)l;
        off16 += (unsigned long long)items + (unsigned long long)large + 2ull * g->wpt * (unsigned long long)tips;
        e += items; t += tips; l += large;
        const int b = b0 + i;
        g->f[b / (NB / 4) + 2] = e;                               // SdbgReader::read_info, sdbg_multi_io.h:253-268
    }
    // a bucket range that ends inside a quarter leaves the later f entries at the running total, like the reader's loop
    for (int q = (b1 - 1) / (NB / 4) + 3; q < 6; ++q) g->f[q] = e;
    if (off16 * 2 != n_bytes) { g->err = "sdbg_append: the bucket table does not add up to n_bytes"; return MGTA_ERR_ARG; }
    int rc;
    // arrays (zero-filled growth: partial words at the seam are completed by atomicOr)
    if ((rc = grow(g, g->w, (size_t)((e + 15) / 16) * 8 + 64, (size_t)((g->n_edges + 15) / 16) * 8))) return rc;
    if ((rc = grow(g, g->last, bit_bytes(e) + 64, bit_bytes(g->n_edges)))) return rc;
    if ((rc = grow(g, g->tip, bit_bytes(e) + 64, bit_bytes(g->n_edges)))) return rc;
    if ((rc = grow(g, g->invalid, bit_bytes(e) + 64, bit_bytes(g->n_edges)))) return rc;
    if (g->need_mult) {
        if ((rc = grow(g, g->edge_multi, (size_t)e + 64, (size_t)g->n_edges))) return rc;
        if ((rc = grow(g, g->large_edge, (size_t)l * 8 + 64, (size_t)g->n_large * 8))) return rc;
        if ((rc = grow(g, g->large_val, (size_t)l * 2 + 64, (size_t)g->n_large * 2))) return rc;
    } else {
        if ((rc = grow(g, g->multi1, bit_bytes(e) + 64, bit_bytes(g->n_edges)))) return rc;
        if ((rc = grow(g, g->large_edge, 64, 0))) return rc;
        if ((rc = grow(g, g->large_val, 64, 0))) return rc;
    }
    if ((rc = grow(g, g->tip_seq, (size_t)t * g->wpt * 4 + 64, (size_t)g->n_tips * g->wpt * 4))) return rc;
    if ((rc = grow(g, g->base, (size_t)n * 32, 0))) return rc;
    if ((rc = grow(g, g->meta, (size_t)n * 24, 0))) return rc;
    SCK(cudaMemcpyAsync(g->base.p, base.data(), (size_t)n * 32, cudaMemcpyHostToDevice, g->stream));
    SCK(cudaMemcpyAsync(g->meta.p, meta, (size_t)n * 24, cudaMemcpyHostToDevice, g->stream));
    const uint16_t *d_stream = nullptr;
    cudaPointerAttributes pa;
    const bool on_device = n_bytes && cudaPointerGetAttributes(&pa, bytes) == cudaSuccess && pa.type == cudaMemoryTypeDevice;
    cudaGetLastError();
    if (on_device) {
        d_stream = reinterpret_cast<const uint16_t *>(bytes);
    } else if (n_bytes) {
        if ((rc = grow(g, g->staging, n_bytes + 64, 0))) return rc;
        SCK(cudaMemcpyAsync(g->staging.p, bytes, n_bytes, cudaMemcpyHostToDevice, g->stream));
        d_stream = reinterpret_cast<const uint16_t *>(g->staging.p);
    }
    if (n_bytes) {
        ParseParams P;
        memset(&P, 0, sizeof(P));
        P.stream = d_stream; P.base = (const unsigned long long *)g->base.p; P.meta = (const long long *)g->meta.p;
        P.n_buckets = n; P.wpt = g->wpt; P.need_mult = g->need_mult;
        P.w = (uint32_t *)g->w.p; P.last = (uint32_t *)g->last.p; P.tip = (uint32_t *)g->tip.p; P.invalid = (uint32_t *)g->invalid.p;
        P.multi1 = g->need_mult ? nullptr : (uint32_t *)g->multi1.p;
        P.edge_multi = (uint8_t *)g->edge_multi.p; P.tip_seq = (uint32_t *)g->tip_seq.p;
        P.large_edge = (unsigned long long *)g->large_edge.p; P.large_val = (uint16_t *)g->large_val.p; P.err = g->d_err;
        const int grid = std::max(1, std::min((n + PARSE_WARPS - 1) / PARSE_WARPS, 148 * 8));
        k_sdbg_parse<<<grid, PARSE_WARPS * 32, 0, g->stream>>>(P);
        SCK(cudaGetLastError());
    }
    SCK(cudaStreamSynchronize(g->stream));                         // base / meta / the caller's bytes may go away after the call
    g->n_edges = e; g->n_tips = t; g->n_large = l;
    return MGTA_OK;
}

namespace {
template <int NC>
int build_rank(mgta_sdbg *g, const void *text, DevBuf &minor, DevBuf &major, long long *freq_host) {
    const long long length = g->n_edges, n_minor = g->n_minor, n_major = g->n_major;
    int rc;
    if ((rc = grow(g, minor, (size_t)NC * n_minor * 2 + 64, 0))) return rc;
    if ((rc = grow(g, major, (size_t)NC * n_major * 8 + 64, 0))) return rc;
    if ((rc = grow(g, g->small, 4096, 0))) return rc;
    long long *d_freq = (long long *)g->small.p;
    SCK(cudaMemsetAsync(major.p, 0, (size_t)NC * n_major * 8, g->stream));
    k_rank_minor<NC><<<(unsigned)n_major, 256, 0, g->stream>>>((const unsigned long long *)text, length, n_minor, (uint16_t *)minor.p,
                                                              (long long *)major.p, n_major);
    k_rank_major<<<NC, 1024, 0, g->stream>>>((long long *)major.p, n_major, d_freq);
    k_rank_close<<<1, 32, 0, g->stream>>>((uint16_t *)minor.p, (const long long *)major.p, d_freq, n_minor, n_major, NC);
    SCK(cudaGetLastError());
    SCK(cudaMemcpyAsync(freq_host, d_freq, NC * 8, cudaMemcpyDeviceToHost, g->stream));
    SCK(cudaStreamSynchronize(g->stream));
    return MGTA_OK;
}

int build_select(mgta_sdbg *g, const DevBuf &minor, const DevBuf &major, int c, long long count, DevBuf &table) {
    const long long n_table = (count + 255) / 256 + 1;
    int rc;
    if ((rc = grow(g, table, (size_t)n_table * 4 + 64, 0))) return rc;
    k_select_table<<<(unsigned)((n_table + 255) / 256), 256, 0, g->stream>>>((const uint16_t *)minor.p + (size_t)c * g->n_minor,
                                                                          (const long long *)major.p + (size_t)c * g->n_major, g->n_minor, count,
                                                                          (uint32_t *)table.p, n_table);
    SCK(cudaGetLastError());
    return MGTA_OK;
}
}  // namespace

extern "C" int mgta_sdbg_finish(mgta_sdbg *g) {
    if (!g) return MGTA_ERR_ARG;
    if (g->finished) return MGTA_OK;
    SCK(cudaSetDevice(g->device));
    unsigned h_err = 0;
    SCK(cudaMemcpyAsync(&h_err, g->d_err, 4, cudaMemcpyDeviceToHost, g->stream));
    SCK(cudaStreamSynchronize(g->stream));
    if (h_err) { char b[128]; snprintf(b, sizeof(b), "sdbg: the record stream does not match its bucket table (flags 0x%x)", h_err); g->err = b; return MGTA_ERR_ARG; }
    int rc;
    if (g->n_edges == 0) {                                          // keep every array addressable
        if ((rc = grow(g, g->w, 64, 0)) || (rc = grow(g, g->last, 64, 0)) || (rc = grow(g, g->tip, 64, 0)) || (rc = grow(g, g->invalid, 64, 0)) ||
            (rc = grow(g, g->edge_multi, 64, 0)) || (rc = grow(g, g->multi1, 64, 0)) || (rc = grow(g, g->tip_seq, 64, 0)) ||
            (rc = grow(g, g->large_edge, 64, 0)) || (rc = grow(g, g->large_val, 64, 0)))
            return rc;
    }
    for (int b = g->next_bucket; b <= NB; ++b) g->bucket_start[b] = g->n_edges;   // buckets no delivery reached
    g->n_minor = (g->n_edges + 255) / 256 + 1;
    g->n_major = (g->n_edges + 65535) / 65536 + 1;
    if ((rc = build_rank<9>(g, g->w.p, g->w_minor, g->w_major, g->w_freq))) return rc;
    if ((rc = build_rank<1>(g, g->last.p, g->last_minor, g->last_major, &g->last_ones))) return rc;
    if ((rc = build_rank<1>(g, g->tip.p, g->tip_minor, g->tip_major, &g->tip_ones))) return rc;
    for (int c = 0; c < 9; ++c)
        if ((rc = build_select(g, g->w_minor, g->w_major, c, g->w_freq[c], g->w_sel[c]))) return rc;
    if ((rc = build_select(g, g->last_minor, g->last_major, 0, g->last_ones, g->last_sel))) return rc;
    // rank_f[i] = rs_last_.Rank(f[i] - 1) = ones in last[0, f[i])  (succinct_dbg.h:73-75; f[0] = -1 reads before the array in
    // the reference and yields 0)
    long long *d_pos = (long long *)g->small.p + 16, *d_out = (long long *)g->small.p + 32;
    SCK(cudaMemcpyAsync(d_pos, g->f, 6 * 8, cudaMemcpyHostToDevice, g->stream));
    k_rank1_at<<<1, 32, 0, g->stream>>>((const unsigned long long *)g->last.p, (const uint16_t *)g->last_minor.p, (const long long *)g->last_major.p,
                                        g->n_edges, g->last_ones, d_pos, d_out, 6);
    SCK(cudaGetLastError());
    SCK(cudaMemcpyAsync(g->rank_f, d_out, 6 * 8, cudaMemcpyDeviceToHost, g->stream));
    SCK(cudaStreamSynchronize(g->stream));
    g->finished = true;
    return MGTA_OK;
}

extern "C" int mgta_sdbg_header(const mgta_sdbg *g, mgta_sdbg_header_t *h) {
    if (!g || !h) return MGTA_ERR_ARG;
    memset(h, 0, sizeof(*h));
    h->size = g->n_edges; h->kmer_k = g->kmer_k; h->num_tips = g->n_tips; h->words_per_tip_label = g->wpt; h->num_large_mul = g->n_large;
    for (int i = 0; i < 6; ++i) { h->f[i] = g->f[i]; h->rank_f[i] = g->rank_f[i]; }
    for (int i = 0; i < 9; ++i) h->w_freq[i] = g->w_freq[i];
    h->last_ones = g->last_ones; h->tip_ones = g->tip_ones;
    h->n_minor = g->n_minor; h->n_major = g->n_major;
    return MGTA_OK;
}

extern "C" int mgta_sdbg_array(mgta_sdbg *g, int which, int c, const void **dev_ptr, uint64_t *n_bytes) {
    if (!g || !dev_ptr || !n_bytes) return MGTA_ERR_ARG;
    const long long n = g->n_edges;
    const size_t wl = bit_bytes(n);
    const void *p = nullptr;
    size_t b = 0;
    const bool tab = which >= MGTA_SDBG_W_MINOR;
    if (tab && !g->finished) { g->err = "sdbg_array: call mgta_sdbg_finish first"; return MGTA_ERR_STATE; }
    if ((which == MGTA_SDBG_W_MINOR || which == MGTA_SDBG_W_MAJOR || which == MGTA_SDBG_W_SELECT) && (c < 0 || c > 8)) return MGTA_ERR_ARG;
    switch (which) {
        case MGTA_SDBG_W: p = g->w.p; b = (size_t)((n + 15) / 16) * 8; break;
        case MGTA_SDBG_LAST: p = g->last.p; b = wl; break;
        case MGTA_SDBG_IS_TIP: p = g->tip.p; b = wl; break;
        case MGTA_SDBG_INVALID: p = g->invalid.p; b = wl; break;
        case MGTA_SDBG_IS_MULTI_1: if (g->need_mult) return MGTA_ERR_ARG; p = g->multi1.p; b = wl; break;
        case MGTA_SDBG_EDGE_MULTI: if (!g->need_mult) return MGTA_ERR_ARG; p = g->edge_multi.p; b = (size_t)n; break;
        case MGTA_SDBG_LARGE_EDGE: p = g->large_edge.p; b = g->need_mult ? (size_t)g->n_large * 8 : 0; break;
        case MGTA_SDBG_LARGE_VALUE: p = g->large_val.p; b = g->need_mult ? (size_t)g->n_large * 2 : 0; break;
        case MGTA_SDBG_TIP_SEQ: p = g->tip_seq.p; b = (size_t)g->n_tips * g->wpt * 4; break;
        case MGTA_SDBG_W_MINOR: p = (const uint16_t *)g->w_minor.p + (size_t)c * g->n_minor; b = (size_t)g->n_minor * 2; break;
        case MGTA_SDBG_W_MAJOR: p = (const long long *)g->w_major.p + (size_t)c * g->n_major; b = (size_t)g->n_major * 8; break;
        case MGTA_SDBG_W_SELECT: p = g->w_sel[c].p; b = (size_t)((g->w_freq[c] + 255) / 256 + 1) * 4; break;
        case MGTA_SDBG_LAST_MINOR: p = g->last_minor.p; b = (size_t)g->n_minor * 2; break;
        case MGTA_SDBG_LAST_MAJOR: p = g->last_major.p; b = (size_t)g->n_major * 8; break;
        case MGTA_SDBG_LAST_SELECT: p = g->last_sel.p; b = (size_t)((g->last_ones + 255) / 256 + 1) * 4; break;
        case MGTA_SDBG_TIP_MINOR: p = g->tip_minor.p; b = (size_t)g->n_minor * 2; break;
        case MGTA_SDBG_TIP_MAJOR: p = g->tip_major.p; b = (size_t)g->n_major * 8; break;
        default: return MGTA_ERR_ARG;
    }
    *dev_ptr = p; *n_bytes = b;
    return MGTA_OK;
}

extern "C" int mgta_sdbg_copy(mgta_sdbg *g, int which, int c, void *host, uint64_t n_bytes) {
    const void *p = nullptr;
    uint64_t b = 0;
    int rc = mgta_sdbg_array(g, which, c, &p, &b);
    if (rc) return rc;
    if (n_bytes < b) { g->err = "sdbg_copy: host buffer too small"; return MGTA_ERR_ARG; }
    SCK(cudaSetDevice(g->device));
    if (b) SCK(cudaMemcpyAsync(host, p, b, cudaMemcpyDeviceToHost, g->stream));
    SCK(cudaStreamSynchronize(g->stream));
    return MGTA_OK;
}

// sink adapter: mgta_stage2(ctx, mgta_sdbg_sink, g, totals) feeds the builder from the stage-2 deliveries
extern "C" int mgta_sdbg_sink(void *user, int32_t b0, int32_t b1, const void *bytes, uint64_t n_bytes, const int64_t *meta) {
    return mgta_sdbg_append((mgta_sdbg *)user, b0, b1, bytes, n_bytes, meta);
}
