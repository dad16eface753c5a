// sdbg_index.cuh -- the device SdBG shared by the index builder (sdbg_index.cu), the navigation queries (sdbg_query.cu) and
// the unitigs (sdbg_unitig.cu): the state behind mgta_sdbg, and the rank arithmetic over its tables (layouts: sdbg_index.cu
// header comment).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <algorithm>
#include <string>
#include <vector>

#include "../../include/mgta_cuda.h"

namespace mgta_sdbg_impl {

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
};

// counts of every character in one u64 of 16 4-bit characters (CountCharInWord_, rank_and_select.h:344-349)
__device__ __forceinline__ int count_char(unsigned long long x, unsigned c) {
    x ^= ~(0x1111111111111111ull * c);
    x &= x >> 2;
    x &= x >> 1;
    return __popcll(x & 0x1111111111111111ull);
}

// number of ones in bits [0, pos) of a bit vector with `length` bits and `total` ones, from its rank tables
// (major: exclusive count every 65536 positions, minor: u16 count relative to the major entry every 256 positions)
__device__ __forceinline__ long long rank1(const unsigned long long *__restrict__ text, const uint16_t *__restrict__ minor,
                                           const long long *__restrict__ major, long long length, long long total, long long pos) {
    if (pos <= 0) return 0;
    if (pos >= length) return total;
    const long long iv = pos / 256;
    long long r = major[iv / 256] + (long long)minor[iv];
    for (long long q = iv * 256; q < pos; q += 64) {
        unsigned long long x = text[q / 64];
        if (pos - q < 64) x &= (1ull << (pos - q)) - 1ull;
        r += __popcll(x);
    }
    return r;
}

}  // namespace mgta_sdbg_impl

struct mgta_sdbg {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int need_mult = 1, kmer_k = 0, wpt = 0;
    bool finished = false;
    std::string err;
    long long n_edges = 0, n_tips = 0, n_large = 0;
    int next_bucket = 0;
    long long f[6] = {-1, 0, 0, 0, 0, 0}, rank_f[6] = {0, 0, 0, 0, 0, 0};
    mgta_sdbg_impl::DevBuf w, last, tip, invalid, multi1, edge_multi, tip_seq, large_edge, large_val, staging, base, meta;
    // tables (finish)
    mgta_sdbg_impl::DevBuf w_minor, w_major, last_minor, last_major, tip_minor, tip_major, w_sel[9], last_sel, small;
    long long w_freq[9] = {0}, last_ones = 0, tip_ones = 0;
    long long n_minor = 0, n_major = 0;
    unsigned *d_err = nullptr;
    // first edge of every lv1 bucket (65536 + 1 entries, from the deliveries' bucket tables), and the queries' buffers
    std::vector<long long> bucket_start = std::vector<long long>(65537, 0);
    mgta_sdbg_impl::DevBuf q_bucket, q_in, q_out, q_err;
    // unitigs (sdbg_unitig.cu): the rows and sequence of the last mgta_sdbg_unitigs, and its scratch (freed when it returns)
    mgta_sdbg_impl::DevBuf ut_rows, ut_seq, ut_edge, ut_seg, ut_jump;
    bool ut_ready = false;
    long long ut_n_rows = 0;
    unsigned long long ut_n_chars = 0;
};

#define SCK(call)                                                                                        \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) {                                                                         \
            char buf_[512];                                                                              \
            snprintf(buf_, sizeof(buf_), "%s:%d: %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            g->err = buf_;                                                                               \
            return MGTA_ERR_CUDA;                                                                        \
        }                                                                                                \
    } while (0)

namespace mgta_sdbg_impl {

// grows a zero-filled device buffer to at least `bytes`, keeping `keep` bytes
inline int grow(mgta_sdbg *g, DevBuf &b, size_t bytes, size_t keep) {
    if (bytes <= b.cap) return MGTA_OK;
    size_t ncap = std::max(bytes, b.cap + b.cap / 2);
    ncap = (ncap + 255) & ~(size_t)255;
    void *np = nullptr;
    SCK(cudaMalloc(&np, ncap));
    if (keep) SCK(cudaMemcpyAsync(np, b.p, keep, cudaMemcpyDeviceToDevice, g->stream));
    SCK(cudaMemsetAsync((char *)np + keep, 0, ncap - keep, g->stream));
    SCK(cudaStreamSynchronize(g->stream));
    cudaFree(b.p);
    b.p = np; b.cap = ncap;
    return MGTA_OK;
}

inline size_t bit_bytes(long long n) { return (size_t)((n + 63) / 64) * 8; }

}  // namespace mgta_sdbg_impl
