// rANS coder kernels + stream sets + bin tables (sm_100a).
//
// Reference being replaced (fhkingma/bitswap @ dfe0bf7d): class ANS, cifar_compress.py:12-67, and the
// float64 logistic table construction around it, cifar_compress.py:182-187,197-202,245-250.
//
// Parallelisation: the reference stream is inherently serial (every symbol-op depends on the previous
// head), so bit-identity forces ONE WARP = ONE STREAM; the 32 lanes split the *bins* of the row being
// coded.  The expensive part -- (S-1) float64 sigmoids per symbol-op, needed because the reference's
// integer quantisation couples every bin of a row (remnant at the row argmax) -- is the part the lanes
// parallelise; the integer head update is done redundantly by all lanes.
#include <stdarg.h>
#include <string.h>
#include <vector>
#include "bsw_common.cuh"

static thread_local char g_err[512] = "";
void bsw_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
extern "C" const char *bsw_last_error(void) { return g_err; }
extern "C" int bsw_version(void) { return 100; }

#define FULL 0xffffffffu

// ================================================================================================
// Stream sets
// ================================================================================================
extern "C" int bsw_streams_create(bsw_streams **out, int n_streams, int64_t capacity_words) {
    BSW_REQUIRE(out && n_streams > 0 && capacity_words > 0, "bsw_streams_create: bad arguments");
    bsw_streams *s = new bsw_streams();
    s->B = n_streams;
    s->cap = (capacity_words + 31) / 32 * 32;
    BSW_CUDA(cudaMalloc(&s->words, sizeof(uint32_t) * s->cap * s->B));
    BSW_CUDA(cudaMalloc(&s->nwords, sizeof(int32_t) * s->B));
    BSW_CUDA(cudaMalloc(&s->heads, sizeof(uint64_t) * s->B));
    BSW_CUDA(cudaMalloc(&s->flags, sizeof(int32_t) * s->B));
    BSW_CUDA(cudaMalloc(&s->minwords, sizeof(int32_t) * s->B));
    BSW_CUDA(cudaMemset(s->minwords, 0, sizeof(int32_t) * s->B));
    BSW_CUDA(cudaMalloc(&s->restwords, sizeof(int32_t) * s->B));
    BSW_CUDA(cudaMemset(s->restwords, 0xff, sizeof(int32_t) * s->B));
    BSW_CUDA(cudaMemset(s->nwords, 0, sizeof(int32_t) * s->B));
    BSW_CUDA(cudaMemset(s->heads, 0, sizeof(uint64_t) * s->B));
    BSW_CUDA(cudaMemset(s->flags, 0, sizeof(int32_t) * s->B));
    *out = s;
    return BSW_OK;
}
extern "C" int bsw_streams_destroy(bsw_streams *s) {
    if (!s) return BSW_OK;
    cudaFree(s->words); cudaFree(s->nwords); cudaFree(s->heads); cudaFree(s->flags); cudaFree(s->minwords); cudaFree(s->restwords);
    delete s;
    return BSW_OK;
}
extern "C" int bsw_streams_count(const bsw_streams *s) { return s ? s->B : 0; }
extern "C" int64_t bsw_streams_capacity(const bsw_streams *s) { return s ? s->cap : 0; }

extern "C" int bsw_streams_import(bsw_streams *s, int first, int count, const uint32_t *words_host,
                                  const int64_t *offsets_host, const uint64_t *heads_host) {
    BSW_REQUIRE(s && first >= 0 && count >= 0 && first + count <= s->B, "bsw_streams_import: range");
    std::vector<int32_t> n(count);
    for (int i = 0; i < count; ++i) {
        int64_t len = offsets_host[i + 1] - offsets_host[i];
        BSW_REQUIRE(len >= 0 && len <= s->cap, "bsw_streams_import: stream longer than capacity");
        n[i] = (int32_t)len;
        if (len)
            BSW_CUDA(cudaMemcpy(s->words + (int64_t)(first + i) * s->cap, words_host + offsets_host[i],
                                sizeof(uint32_t) * len, cudaMemcpyHostToDevice));
    }
    BSW_CUDA(cudaMemcpy(s->nwords + first, n.data(), sizeof(int32_t) * count, cudaMemcpyHostToDevice));
    BSW_CUDA(cudaMemcpy(s->minwords + first, n.data(), sizeof(int32_t) * count, cudaMemcpyHostToDevice));
    BSW_CUDA(cudaMemcpy(s->heads + first, heads_host, sizeof(uint64_t) * count, cudaMemcpyHostToDevice));
    BSW_CUDA(cudaMemset(s->flags + first, 0, sizeof(int32_t) * count));
    BSW_CUDA(cudaMemset(s->restwords + first, 0xff, sizeof(int32_t) * count));
    return BSW_OK;
}

__global__ void k_streams_fill(bsw_streams sv, const uint32_t *src, int64_t n, uint64_t head) {
    int b = blockIdx.y;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        sv.words[(int64_t)b * sv.cap + i] = src[i];
    if (blockIdx.x == 0 && threadIdx.x == 0) { sv.nwords[b] = (int32_t)n; sv.minwords[b] = (int32_t)n; sv.restwords[b] = -1; sv.heads[b] = head; sv.flags[b] = 0; }
}
extern "C" int bsw_streams_fill(bsw_streams *s, const uint32_t *words_host, int64_t nwords, uint64_t head) {
    BSW_REQUIRE(s && nwords >= 0 && nwords <= s->cap, "bsw_streams_fill: nwords exceeds capacity");
    uint32_t *tmp = nullptr;
    BSW_CUDA(cudaMalloc(&tmp, sizeof(uint32_t) * (nwords ? nwords : 1)));
    if (nwords) BSW_CUDA(cudaMemcpy(tmp, words_host, sizeof(uint32_t) * nwords, cudaMemcpyHostToDevice));
    dim3 grid((unsigned)((nwords + 255) / 256 > 0 ? (nwords + 255) / 256 : 1), s->B);
    if (grid.x > 64) grid.x = 64;
    k_streams_fill<<<grid, 256>>>(*s, tmp, nwords, head);
    BSW_LAUNCH_CHECK();
    BSW_CUDA(cudaDeviceSynchronize());
    cudaFree(tmp);
    return BSW_OK;
}
extern "C" int bsw_streams_sizes(bsw_streams *s, int64_t *nwords_host, uint64_t *heads_host, int32_t *flags_host) {
    BSW_REQUIRE(s, "null stream set");
    BSW_CUDA(cudaDeviceSynchronize());
    if (nwords_host) {
        std::vector<int32_t> n(s->B);
        BSW_CUDA(cudaMemcpy(n.data(), s->nwords, sizeof(int32_t) * s->B, cudaMemcpyDeviceToHost));
        for (int i = 0; i < s->B; ++i) nwords_host[i] = n[i];
    }
    if (heads_host) BSW_CUDA(cudaMemcpy(heads_host, s->heads, sizeof(uint64_t) * s->B, cudaMemcpyDeviceToHost));
    if (flags_host) BSW_CUDA(cudaMemcpy(flags_host, s->flags, sizeof(int32_t) * s->B, cudaMemcpyDeviceToHost));
    return BSW_OK;
}
extern "C" int bsw_streams_min_words(bsw_streams *s, int64_t *min_host) {
    BSW_REQUIRE(s && min_host, "null argument");
    BSW_CUDA(cudaDeviceSynchronize());
    std::vector<int32_t> n(s->B);
    BSW_CUDA(cudaMemcpy(n.data(), s->minwords, sizeof(int32_t) * s->B, cudaMemcpyDeviceToHost));
    for (int i = 0; i < s->B; ++i) min_host[i] = n[i];
    return BSW_OK;
}
// a12 accounting: the word count right after a chain's first pop, the reference's len(restbits) - 1 (cifar_compress.py:190-192,254)
__global__ void k_mark_rest(bsw_streams sv, int first, int count) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count && sv.restwords[first + i] < 0) sv.restwords[first + i] = sv.nwords[first + i];
}
int bsw_streams_mark_rest(bsw_streams *s, int first, int count, cudaStream_t st) {
    k_mark_rest<<<(count + 255) / 256, 256, 0, st>>>(*s, first, count);
    BSW_LAUNCH_CHECK();
    return BSW_OK;
}
extern "C" int bsw_streams_rest_words(bsw_streams *s, int64_t *rest_host) {
    BSW_REQUIRE(s && rest_host, "null argument");
    BSW_CUDA(cudaDeviceSynchronize());
    std::vector<int32_t> n(s->B);
    BSW_CUDA(cudaMemcpy(n.data(), s->restwords, sizeof(int32_t) * s->B, cudaMemcpyDeviceToHost));
    for (int i = 0; i < s->B; ++i) rest_host[i] = n[i];
    return BSW_OK;
}
extern "C" int bsw_streams_export(bsw_streams *s, int first, int count, uint32_t *words_host,
                                  const int64_t *offsets_host) {
    BSW_REQUIRE(s && first >= 0 && count >= 0 && first + count <= s->B, "bsw_streams_export: range");
    std::vector<int32_t> n(count);
    BSW_CUDA(cudaMemcpy(n.data(), s->nwords + first, sizeof(int32_t) * count, cudaMemcpyDeviceToHost));
    for (int i = 0; i < count; ++i)
        if (n[i])
            BSW_CUDA(cudaMemcpy(words_host + offsets_host[i], s->words + (int64_t)(first + i) * s->cap,
                                sizeof(uint32_t) * n[i], cudaMemcpyDeviceToHost));
    return BSW_OK;
}
// ---- packed (de)serialisation: every stream's words gathered into / scattered from ONE contiguous device buffer with
// coalesced 128-byte warp accesses, so a host export/import is three memcpys instead of two per stream.
// Trimmed form (base != NULL): only words[base_b .. n_b) travel, base_b = the lowest depth the stack ever reached -- the
// initial random words below it were never borrowed and the receiver already has them (demo_compress.py:137,160
// `excess_state_len`; the receiver re-creates them from the seed, demo_decompress.py:176-186).
__global__ void k_pack_offsets(const int32_t *__restrict__ n, const int32_t *__restrict__ minw, int trim, int count,
                               int64_t *__restrict__ offs, int32_t *__restrict__ base_out) {
    // single block exclusive scan (count <= a few 10^4 streams)
    __shared__ long long carry;
    __shared__ long long part[32];
    if (threadIdx.x == 0) { carry = 0; offs[0] = 0; }
    __syncthreads();
    for (int base = 0; base < count; base += blockDim.x) {
        int i = base + threadIdx.x;
        int lo = (trim && i < count) ? min(minw[i], n[i]) : 0;
        if (base_out && i < count) base_out[i] = lo;
        long long v = i < count ? n[i] - lo : 0, x = v;
        for (int o = 1; o < 32; o <<= 1) { long long t = __shfl_up_sync(FULL, x, o); if ((threadIdx.x & 31) >= o) x += t; }
        if ((threadIdx.x & 31) == 31) part[threadIdx.x >> 5] = x;
        __syncthreads();
        if (threadIdx.x < 32) {
            long long p = threadIdx.x < (blockDim.x >> 5) ? part[threadIdx.x] : 0, y = p;
            for (int o = 1; o < 32; o <<= 1) { long long t = __shfl_up_sync(FULL, y, o); if (threadIdx.x >= o) y += t; }
            part[threadIdx.x] = y - p;
        }
        __syncthreads();
        long long incl = x + part[threadIdx.x >> 5] + carry;
        if (i < count) offs[i + 1] = incl;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) carry = incl;
        __syncthreads();
    }
}
__global__ void k_pack_words(bsw_streams sv, int first, const int64_t *__restrict__ offs, const int32_t *__restrict__ base,
                             uint32_t *__restrict__ out, uint64_t *__restrict__ heads_out) {
    int b = blockIdx.x;
    const int lo = base ? base[b] : 0;
    const uint32_t *src = sv.words + (int64_t)(first + b) * sv.cap + lo;
    int n = sv.nwords[first + b] - lo;
    uint32_t *dst = out + offs[b];
    for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
    if (threadIdx.x == 0) heads_out[b] = sv.heads[first + b];
}
__global__ void k_unpack_words(bsw_streams sv, int first, const int64_t *__restrict__ offs, const int32_t *__restrict__ base,
                               const uint32_t *__restrict__ in, const uint64_t *__restrict__ heads_in) {
    int b = blockIdx.x;
    const int lo = base ? base[b] : 0;
    int64_t o = offs[b];
    int n = (int)(offs[b + 1] - o);
    if ((int64_t)lo + n > sv.cap) {                       // corrupt lengths must not write past the stream's row
        if (threadIdx.x == 0) sv.flags[first + b] = BSW_E_OVERFLOW;
        return;
    }
    uint32_t *dst = sv.words + (int64_t)(first + b) * sv.cap + lo;
    for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = in[o + i];
    if (threadIdx.x == 0) {
        sv.nwords[first + b] = lo + n; sv.minwords[first + b] = base ? lo : n; sv.heads[first + b] = heads_in[b]; sv.flags[first + b] = 0;
    }
}
static int pack_impl(bsw_streams *s, int first, int count, uint32_t *words_dev, int64_t *offsets_dev, uint64_t *heads_dev,
                     int32_t *base_dev, void *stream) {
    BSW_REQUIRE(s && first >= 0 && count > 0 && first + count <= s->B && words_dev && offsets_dev && heads_dev, "bsw_streams_pack: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    k_pack_offsets<<<1, 1024, 0, st>>>(s->nwords + first, s->minwords + first, base_dev != nullptr, count, offsets_dev, base_dev);
    BSW_LAUNCH_CHECK();
    k_pack_words<<<count, 256, 0, st>>>(*s, first, offsets_dev, base_dev, words_dev, heads_dev);
    BSW_LAUNCH_CHECK();
    return BSW_OK;
}
extern "C" int bsw_streams_pack(bsw_streams *s, int first, int count, uint32_t *words_dev, int64_t *offsets_dev,
                                uint64_t *heads_dev, void *stream) {
    return pack_impl(s, first, count, words_dev, offsets_dev, heads_dev, nullptr, stream);
}
extern "C" int bsw_streams_pack_trimmed(bsw_streams *s, int first, int count, uint32_t *words_dev, int64_t *offsets_dev,
                                        uint64_t *heads_dev, int32_t *base_dev, void *stream) {
    BSW_REQUIRE(base_dev, "bsw_streams_pack_trimmed: base_dev is required");
    return pack_impl(s, first, count, words_dev, offsets_dev, heads_dev, base_dev, stream);
}
extern "C" int bsw_streams_unpack(bsw_streams *s, int first, int count, const uint32_t *words_dev, const int64_t *offsets_dev,
                                  const uint64_t *heads_dev, void *stream) {
    BSW_REQUIRE(s && first >= 0 && count > 0 && first + count <= s->B && words_dev && offsets_dev && heads_dev, "bsw_streams_unpack: bad arguments");
    k_unpack_words<<<count, 256, 0, (cudaStream_t)stream>>>(*s, first, offsets_dev, nullptr, words_dev, heads_dev);
    BSW_LAUNCH_CHECK();
    return BSW_OK;
}
extern "C" int bsw_streams_unpack_trimmed(bsw_streams *s, int first, int count, const uint32_t *words_dev, const int64_t *offsets_dev,
                                          const uint64_t *heads_dev, const int32_t *base_dev, void *stream) {
    BSW_REQUIRE(s && first >= 0 && count > 0 && first + count <= s->B && words_dev && offsets_dev && heads_dev && base_dev, "bsw_streams_unpack_trimmed: bad arguments");
    k_unpack_words<<<count, 256, 0, (cudaStream_t)stream>>>(*s, first, offsets_dev, base_dev, words_dev, heads_dev);
    BSW_LAUNCH_CHECK();
    return BSW_OK;
}

extern "C" int bsw_streams_device_ptrs(bsw_streams *s, uint32_t **w, int32_t **n, uint64_t **h, int32_t **f) {
    BSW_REQUIRE(s, "null stream set");
    if (w) *w = s->words;
    if (n) *n = s->nwords;
    if (h) *h = s->heads;
    if (f) *f = s->flags;
    return BSW_OK;
}
__global__ void k_total_words(const int32_t *n, int B, int64_t *out) {
    __shared__ long long part[32];
    long long v = 0;
    for (int i = threadIdx.x; i < B; i += blockDim.x) v += n[i];
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x < 32) {
        v = threadIdx.x < (blockDim.x >> 5) ? part[threadIdx.x] : 0;
        for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
        if (threadIdx.x == 0) *out = v;
    }
}
extern "C" int bsw_streams_total_words(bsw_streams *s, int64_t *total_dev, void *stream) {
    BSW_REQUIRE(s && total_dev, "null argument");
    k_total_words<<<1, 1024, 0, (cudaStream_t)stream>>>(s->nwords, s->B, total_dev);
    BSW_LAUNCH_CHECK();
    return BSW_OK;
}

// ================================================================================================
// Warp-level helpers shared by the coder kernels
// ================================================================================================
// Per-warp view of one stream with a 32-word register window over the top of the stack, so that the
// renormalisation words move to/from HBM as whole 128-byte lines.
struct WarpStream {
    uint32_t *words;   // this stream's row
    uint64_t x;        // head (replicated in all lanes)
    int len, cap;
    int wbase;         // index of the word lane 0 holds (multiple of 32), or -1
    uint32_t wbuf;     // lane j holds words[wbase + j]
    int err;

    __device__ __forceinline__ void open(const bsw_streams &sv, int b) {
        words = sv.words + (int64_t)b * sv.cap;
        x = sv.heads[b];
        len = sv.nwords[b];
        cap = (int)sv.cap;
        err = sv.flags[b];
        wbase = -1;
        wbuf = 0;
    }
    __device__ __forceinline__ void close(const bsw_streams &sv, int b, int lane) {
        if (lane == 0) { sv.heads[b] = x; sv.nwords[b] = len; sv.flags[b] = err; if (len < sv.minwords[b]) sv.minwords[b] = len; }
    }
    // ---- pop side: window slides downward -------------------------------------------------------
    __device__ __forceinline__ uint32_t pop_word(int lane) {     // caller guarantees len > 0
        int idx = len - 1;
        if (wbase < 0 || idx < wbase) {
            wbase = idx & ~31;
            wbuf = words[wbase + lane];
        }
        len = idx;
        return __shfl_sync(FULL, wbuf, idx - wbase);
    }
    // ---- push side: window slides upward --------------------------------------------------------
    __device__ __forceinline__ void push_begin(int lane) {
        wbase = len & ~31;
        wbuf = (wbase + lane < len) ? words[wbase + lane] : 0u;
    }
    __device__ __forceinline__ void push_word(uint32_t w, int lane) {   // caller guarantees len < cap
        if (lane == len - wbase) wbuf = w;
        ++len;
        if (len - wbase == 32) {
            words[wbase + lane] = wbuf;
            wbase += 32;
        }
    }
    __device__ __forceinline__ void push_end(int lane) {
        if (lane < len - wbase) words[wbase + lane] = wbuf;
    }
    // ---- the integer recurrences (cifar_compress.py:51-54 and :60-65) -------------------------------
    __device__ __forceinline__ void encode(uint32_t p, uint32_t c, int bits, int lane) {
        uint64_t lim = ((((uint64_t)1 << 32) >> bits) << 32) * (uint64_t)p;
        if (x >= lim) {
            if (len >= cap) { err = BSW_E_OVERFLOW; return; }
            push_word((uint32_t)x, lane);
            x >>= 32;
        }
        uint64_t qd = x / p;
        uint64_t rm = x - qd * p;
        x = (qd << bits) + rm + c;
    }
    __device__ __forceinline__ void decode(uint32_t p, uint32_t c, uint32_t m, int bits, int lane) {
        x = (uint64_t)p * (x >> bits) + m - c;
        if (x < ((uint64_t)1 << 32)) {
            if (len <= 0) { err = BSW_E_UNDERFLOW; return; }
            uint32_t w = pop_word(lane);
            x = (x << 32) | w;
        }
    }
};

__device__ __forceinline__ uint32_t warp_sum_u32(uint32_t v) {
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
__device__ __forceinline__ uint32_t warp_incl_scan_u32(uint32_t v, int lane) {
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(FULL, v, o);
        if (lane >= o) v += t;
    }
    return v;
}
// argmax with the reference's tie rule (first index wins, cifar_compress.py:35 / torch.argmax)
__device__ __forceinline__ void warp_argmax(uint32_t &val, int &idx) {
    for (int o = 16; o; o >>= 1) {
        uint32_t ov = __shfl_xor_sync(FULL, val, o);
        int oi = __shfl_xor_sync(FULL, idx, o);
        if (ov > val || (ov == val && oi < idx)) { val = ov; idx = oi; }
    }
}

// ================================================================================================
// a1: ANS.__init__ -- float64 pmfs -> integer tables (any S).  One warp per row.
// ================================================================================================
__global__ void k_tables_from_pmfs(const double *__restrict__ pmfs, int64_t L, int S, int bits, int q,
                                   uint32_t *__restrict__ P, uint32_t *__restrict__ C, int32_t *err) {
    int lane = threadIdx.x & 31;
    int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= L) return;
    const double *pm = pmfs + row * S;
    uint32_t *Pr = P + row * S, *Cr = C + row * (S + 1);
    const double mult = (double)(((int64_t)1 << bits) - ((int64_t)1 << q));     // cifar_compress.py:28
    // pass 1: sum and first argmax
    uint32_t sum = 0, best = 0;
    int bi = 0x7fffffff;
    for (int k = lane; k < S; k += 32) {
        uint32_t v = (uint32_t)__double2ll_rz(__dmul_rn(pm[k], mult)) + 1u;     // :29 trunc, :32 +1
        sum += v;
        if (v > best) { best = v; bi = k; }
    }
    sum = warp_sum_u32(sum);
    warp_argmax(best, bi);
    uint32_t rem = (1u << bits) - sum;                                          // :35
    // pass 2: cumulative sums
    uint32_t carry = 0;
    if (lane == 0) Cr[0] = 0;
    for (int k0 = 0; k0 < S; k0 += 32) {
        int k = k0 + lane;
        uint32_t v = 0;
        if (k < S) {
            v = (uint32_t)__double2ll_rz(__dmul_rn(pm[k], mult)) + 1u;
            if (k == bi) v += rem;
            Pr[k] = v;
        }
        uint32_t inc = warp_incl_scan_u32(v, lane) + carry;
        if (k < S) Cr[k + 1] = inc;
        carry = __shfl_sync(FULL, inc, 31);
    }
    if (lane == 0 && err && (carry != (1u << bits) || (int32_t)(best + rem) <= 0)) *err = BSW_E_BADTABLE;   // :46
}
extern "C" int bsw_ans_tables(const double *pmfs, int64_t L, int S, int bits, int q, uint32_t *P, uint32_t *C,
                              int32_t *err, void *stream) {
    BSW_REQUIRE(pmfs && P && C && L > 0 && S > 1 && bits > 0 && bits <= 31 && q >= 0 && q < bits, "bsw_ans_tables: bad arguments");
    const int wpb = 8;
    k_tables_from_pmfs<<<(unsigned)((L + wpb - 1) / wpb), wpb * 32, 0, (cudaStream_t)stream>>>(pmfs, L, S, bits, q, P, C, err);
    BSW_LAUNCH_CHECK();
    return BSW_OK;
}

// ================================================================================================
// a4 (export path): logistic pmfs in float64, and a4+a1 materialised tables (shared tables, e.g. prior)
// ================================================================================================
__global__ void k_logistic_pmfs(const double *__restrict__ endp, int64_t ers, const double *__restrict__ mu,
                                const double *__restrict__ sc, int64_t ms, int64_t L, int S, double *__restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= L * S) return;
    int64_t r = i / S;
    int k = (int)(i - r * S);
    const double *e = endp + r * ers;
    double m = mu[r * ms], s = sc[r * ms];
    double chi = (k < S - 1) ? bsw_cdf_div(e[k], m, s) : 1.0;
    double clo = (k > 0) ? bsw_cdf_div(e[k - 1], m, s) : 0.0;
    out[i] = __dsub_rn(chi, clo);      // k==0: c0 - 0 == c0 ; k==S-1: 1.0 - c_{S-2}   (cifar_compress.py:183-184)
}
extern "C" int bsw_logistic_pmfs(const double *endp, int64_t ers, const double *mu, const double *sc, int64_t ms,
                                 int64_t L, int S, double *out, void *stream) {
    BSW_REQUIRE(endp && mu && sc && out && L > 0 && S > 1, "bsw_logistic_pmfs: bad arguments");
    int64_t n = L * S;
    k_logistic_pmfs<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(endp, ers, mu, sc, ms, L, S, out);
    BSW_LAUNCH_CHECK();
    return BSW_OK;
}

__global__ void k_logistic_tables(const double *__restrict__ endp, int64_t ers, const double *__restrict__ mu,
                                  const double *__restrict__ sc, int64_t ms, int64_t L, int S, int bits, int q,
                                  uint32_t *__restrict__ P, uint32_t *__restrict__ C) {
    int lane = threadIdx.x & 31;
    int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= L) return;
    const double *e = endp + row * ers;
    double m = mu[row * ms], s = sc[row * ms];
    uint32_t *Pr = P + row * S, *Cr = C + row * (S + 1);
    const double mult = (double)(((int64_t)1 << bits) - ((int64_t)1 << q));
    auto pk = [&](int k) -> uint32_t {
        double chi = (k < S - 1) ? bsw_cdf_div(e[k], m, s) : 1.0;
        double clo = (k > 0) ? bsw_cdf_div(e[k - 1], m, s) : 0.0;
        return (uint32_t)__double2ll_rz(__dmul_rn(__dsub_rn(chi, clo), mult)) + 1u;
    };
    uint32_t sum = 0, best = 0;
    int bi = 0x7fffffff;
    for (int k = lane; k < S; k += 32) {
        uint32_t v = pk(k);
        Pr[k] = v;
        sum += v;
        if (v > best) { best = v; bi = k; }
    }
    sum = warp_sum_u32(sum);
    warp_argmax(best, bi);
    uint32_t rem = (1u << bits) - sum;
    __syncwarp();
    uint32_t carry = 0;
    if (lane == 0) Cr[0] = 0;
    for (int k0 = 0; k0 < S; k0 += 32) {
        int k = k0 + lane;
        uint32_t v = 0;
        if (k < S) {
            v = Pr[k];
            if (k == bi) { v += rem; Pr[k] = v; }
        }
        uint32_t inc = warp_incl_scan_u32(v, lane) + carry;
        if (k < S) Cr[k + 1] = inc;
        carry = __shfl_sync(FULL, inc, 31);
    }
}
extern "C" int bsw_logistic_tables(const double *endp, int64_t ers, const double *mu, const double *sc, int64_t ms,
                                   int64_t L, int S, int bits, int q, uint32_t *P, uint32_t *C, void *stream) {
    BSW_REQUIRE(endp && mu && sc && P && C && L > 0 && S > 1, "bsw_logistic_tables: bad arguments");
    const int wpb = 8;
    k_logistic_tables<<<(unsigned)((L + wpb - 1) / wpb), wpb * 32, 0, (cudaStream_t)stream>>>(endp, ers, mu, sc, ms, L, S, bits, q, P, C);
    BSW_LAUNCH_CHECK();
    return BSW_OK;
}

// ================================================================================================
// a2/a3 over given integer tables.  One warp per stream.  HBM traffic per symbol-op:
// push 8 B table + 4 B symbol (+ words); pop two 128 B probes of the C row + 8 B + 4 B symbol.
// ================================================================================================
constexpr int TW = 4;   // warps (= streams) per CTA for the table-driven kernels

template <typename SymT>
__global__ void __launch_bounds__(TW * 32) k_push_tables(bsw_streams sv, int first, int count,
        const uint32_t *__restrict__ P, const uint32_t *__restrict__ C, int64_t pss, int64_t css,
        const SymT *__restrict__ sym, int64_t L, int S, int bits) {
    int lane = threadIdx.x & 31;
    int si = blockIdx.x * TW + (threadIdx.x >> 5);
    if (si >= count) return;
    int b = first + si;
    WarpStream ws;
    ws.open(sv, b);
    if (ws.err) return;
    ws.push_begin(lane);
    const uint32_t *Pb = P + (int64_t)si * pss, *Cb = C + (int64_t)si * css;
    const SymT *sy = sym + (int64_t)si * L;
    for (int64_t i0 = 0; i0 < L && !ws.err; i0 += 32) {
        int64_t i = i0 + lane;
        uint32_t p = 1, c = 0;
        if (i < L) {
            int s = (int)sy[i];
            if ((unsigned)s < (unsigned)S) {
                p = Pb[i * S + s];
                c = Cb[i * (S + 1) + s];
            } else p = 0;                                  // symbol outside the support: no table read; flagged below
        }
        int n = (int)min((int64_t)32, L - i0);
        for (int j = 0; j < n && !ws.err; ++j) {
            const uint32_t pj = __shfl_sync(FULL, p, j);
            if (pj == 0u) { ws.err = BSW_E_INVALID; break; }   // the reference raises IndexError at self.pmfs[i, s] (:50)
            ws.encode(pj, __shfl_sync(FULL, c, j), bits, lane);
        }
    }
    ws.push_end(lane);
    ws.close(sv, b, lane);
}

template <typename SymT>
__global__ void __launch_bounds__(TW * 32) k_pop_tables(bsw_streams sv, int first, int count,
        const uint32_t *__restrict__ P, const uint32_t *__restrict__ C, int64_t pss, int64_t css,
        SymT *__restrict__ sym, int64_t L, int S, int bits) {
    int lane = threadIdx.x & 31;
    int si = blockIdx.x * TW + (threadIdx.x >> 5);
    if (si >= count) return;
    int b = first + si;
    WarpStream ws;
    ws.open(sv, b);
    if (ws.err) return;
    const uint32_t *Pb = P + (int64_t)si * pss, *Cb = C + (int64_t)si * css;
    SymT *sy = sym + (int64_t)si * L;
    const uint32_t mask = (uint32_t)(((uint64_t)1 << bits) - 1);
    const int step = (S + 31) / 32;
    for (int64_t i = L - 1; i >= 0 && !ws.err; --i) {
        const uint32_t *Cr = Cb + i * (S + 1);
        uint32_t m = (uint32_t)ws.x & mask;                                     // :60
        // s = max{k : C[k] <= m}  (:61 searchsorted(..., 'right') - 1), two-level ballot search
        int kc = lane * step;
        unsigned bal = __ballot_sync(FULL, kc < S && Cr[kc] <= m);
        int chunk = 31 - __clz(bal);                                            // C[0] = 0 <= m always
        int cnt = 0;
        for (int t0 = 0; t0 < step; t0 += 32) {
            int k = chunk * step + t0 + lane;
            cnt += __popc(__ballot_sync(FULL, (t0 + lane) < step && k < S && Cr[k] <= m));
        }
        int s = chunk * step + cnt - 1;
        if (lane == 0) sy[i] = (SymT)s;                                               // :62
        ws.decode(Pb[i * S + s], Cr[s], m, bits, lane);                         // :63-65
    }
    ws.close(sv, b, lane);
}

static int check_range(bsw_streams *s, int first, int count) {
    BSW_REQUIRE(s && first >= 0 && count > 0 && first + count <= s->B, "stream range out of bounds");
    return BSW_OK;
}
extern "C" int bsw_ans_push(bsw_streams *s, int first, int count, const uint32_t *P, const uint32_t *C, int64_t pss,
                            int64_t css, const int32_t *sym, int64_t L, int S, int bits, void *stream) {
    if (int rc = check_range(s, first, count)) return rc;
    BSW_REQUIRE(P && C && sym && L > 0 && S > 1 && bits > 0 && bits <= 31, "bsw_ans_push: bad arguments");
    k_push_tables<int32_t><<<(count + TW - 1) / TW, TW * 32, 0, (cudaStream_t)stream>>>(*s, first, count, P, C, pss, css, sym, L, S, bits);
    BSW_LAUNCH_CHECK();
    return BSW_OK;
}
extern "C" int bsw_ans_pop(bsw_streams *s, int first, int count, const uint32_t *P, const uint32_t *C, int64_t pss,
                           int64_t css, int32_t *sym, int64_t L, int S, int bits, void *stream) {
    if (int rc = check_range(s, first, count)) return rc;
    BSW_REQUIRE(P && C && sym && L > 0 && S > 1 && bits > 0 && bits <= 31, "bsw_ans_pop: bad arguments");
    k_pop_tables<int32_t><<<(count + TW - 1) / TW, TW * 32, 0, (cudaStream_t)stream>>>(*s, first, count, P, C, pss, css, sym, L, S, bits);
    BSW_LAUNCH_CHECK();
    return BSW_OK;
}

// int16-symbol variants used by the device-resident codec (codec.cu) for the shared prior table
int bsw_ans_push_i16(bsw_streams *s, int first, int count, const uint32_t *P, const uint32_t *C, int64_t pss, int64_t css,
                     const int16_t *sym, int64_t L, int S, int bits, cudaStream_t st) {
    if (int rc = check_range(s, first, count)) return rc;
    k_push_tables<int16_t><<<(count + TW - 1) / TW, TW * 32, 0, st>>>(*s, first, count, P, C, pss, css, sym, L, S, bits);
    BSW_LAUNCH_CHECK();
    return BSW_OK;
}
int bsw_ans_pop_i16(bsw_streams *s, int first, int count, const uint32_t *P, const uint32_t *C, int64_t pss, int64_t css,
                    int16_t *sym, int64_t L, int S, int bits, cudaStream_t st) {
    if (int rc = check_range(s, first, count)) return rc;
    k_pop_tables<int16_t><<<(count + TW - 1) / TW, TW * 32, 0, st>>>(*s, first, count, P, C, pss, css, sym, L, S, bits);
    BSW_LAUNCH_CHECK();
    return BSW_OK;
}

// ================================================================================================
// Fused hot kernels: logistic table in registers + coder.  One warp per stream, lane owns the NB
// consecutive bins [lane*NB, lane*NB+NB) of the row (S = 32*NB).
//
// Per row and warp: S-1 float64 sigmoids (~40 FP64-pipe instructions each) -- the kernel is bound by
// the FP64 pipe, not by HBM (DESIGN.md "ANS kernel roofline").  Endpoint rows are shared by every
// stream; they are brought into a per-warp, bank-conflict-free padded shared-memory tile with
// cp.async one row ahead of the arithmetic.
// ================================================================================================
constexpr int FW = 4;   // warps (= streams) per CTA

template <int NB>
struct RowTable {
    uint32_t P[NB];     // final integer pmf of my bins (remnant applied)
    uint32_t base;      // integer cdf at my first bin
};

__device__ __forceinline__ void cp_async8(void *smem_dst, const void *gsrc) {
    unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(d), "l"(gsrc));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;\n" ::: "memory"); }

// padded tile index of bin k: lane-blocked reads (k = lane*NB + j) and row-interleaved writes
// (k = r*32 + lane) are both bank-conflict free for 8-byte words because NB+1 is odd.
template <int NB>
__device__ __forceinline__ int tile_idx(int k) { return k + k / NB; }
template <int NB>
__host__ __device__ constexpr int tile_doubles() { return 32 * NB + 32; }

template <int NB>
__device__ __forceinline__ void stage_row(double *tile, const double *grow, int lane) {
#pragma unroll
    for (int r = 0; r < NB; ++r) {
        int k = r * 32 + lane;
        cp_async8(tile + tile_idx<NB>(k), grow + k);
    }
}

// Builds the row's integer table (ANS.__init__ semantics) from e[NB] (my endpoints, e[k] = upper
// endpoint of bin k; the last bin of the row has none).
template <int NB>
__device__ __forceinline__ void build_row(const double (&e)[NB], float muf, float scf, double mult, int bits,
                                          int lane, RowTable<NB> &T) {
    const double mu = (double)muf, sc = (double)scf;     // model/cifar_train.py:375-376 up-cast
    const double rsc = __ddiv_rn(1.0, sc);
    // cdf at my last endpoint first: the next lane needs it as its lower neighbour
    double c_last = (lane == 31) ? 1.0 : bsw_cdf_rcp(e[NB - 1], mu, sc, rsc);
    double up = __shfl_up_sync(FULL, c_last, 1);
    double prev = (lane == 0) ? 0.0 : up;
    uint32_t lsum = 0, lbest = 0;
    int lbi = 0;
#pragma unroll
    for (int j = 0; j < NB; ++j) {
        double c = (j == NB - 1) ? c_last : bsw_cdf_rcp(e[j], mu, sc, rsc);
        double pmf = __dsub_rn(c, prev);                                        // cifar_compress.py:183-184
        prev = c;
        uint32_t v = (uint32_t)__double2ll_rz(__dmul_rn(pmf, mult)) + 1u;       // :29, :32
        T.P[j] = v;
        lsum += v;
        if (v > lbest) { lbest = v; lbi = j; }                                  // first maximum within the lane
    }
    uint32_t incl = warp_incl_scan_u32(lsum, lane);
    uint32_t total = __shfl_sync(FULL, incl, 31);
    int bi = lane * NB + lbi;
    warp_argmax(lbest, bi);                                                     // :35 first maximum of the row
    uint32_t rem = (1u << bits) - total;
    T.base = incl - lsum + ((lane * NB > bi) ? rem : 0u);
#pragma unroll
    for (int j = 0; j < NB; ++j)
        if (lane * NB + j == bi) T.P[j] += rem;
}

template <int NB>
__device__ __forceinline__ void load_tile_row(double (&e)[NB], const double *tile, int lane) {
#pragma unroll
    for (int j = 0; j < NB; ++j) e[j] = tile[lane * (NB + 1) + j];
}

// MASK: rowmask holds L/32 words per stream; a clear bit (i & 31) of word i/32 skips row i (template flag: the unmasked
// loop is the plain one)
template <int NB, bool MASK>
__global__ void __launch_bounds__(FW * 32) k_logistic_pop(bsw_streams sv, int first, int count,
        const float *__restrict__ mu, int64_t mss, const float *__restrict__ sc, int64_t sss,
        const double *__restrict__ endp, int64_t ers, int16_t *__restrict__ sym, int64_t L, int bits, int q,
        const uint32_t *__restrict__ rowmask) {
    extern __shared__ double smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int si = blockIdx.x * FW + warp;
    if (si >= count) return;
    int b = first + si;
    WarpStream ws;
    ws.open(sv, b);
    if (ws.err) return;
    const uint32_t *rm = MASK ? rowmask + (int64_t)si * (L >> 5) : nullptr;
    uint32_t live = FULL;              // row mask word of the current block of 32 rows (NULL mask: every row)
    double *tile0 = smem + (size_t)warp * 2 * tile_doubles<NB>();
    double *tile1 = tile0 + tile_doubles<NB>();
    const float *mub = mu + (int64_t)si * mss, *scb = sc + (int64_t)si * sss;
    int16_t *sy = sym + (int64_t)si * L;
    const double mult = (double)(((int64_t)1 << bits) - ((int64_t)1 << q));
    const uint32_t mask = (uint32_t)(((uint64_t)1 << bits) - 1);
    const bool shared_row = (ers == 0);

    double e[NB];
    stage_row<NB>(tile0, endp + (L - 1) * ers, lane);
    cp_async_commit();
    float mu_w = 0.f, sc_w = 1.f;      // lane j holds mu/scale of row (blk*32 + j)
    int my_sym = 0;
    int cur = 0;
    for (int64_t i = L - 1; i >= 0; --i) {
        int j32 = (int)(i & 31);
        if (j32 == 31 || i == L - 1) {                 // new block of 32 rows: coalesced loads
            int64_t r = (i & ~(int64_t)31) + lane;
            mu_w = r < L ? mub[r] : 0.f;
            sc_w = r < L ? scb[r] : 1.f;
            if (MASK) live = __ldg(rm + (i >> 5));
        }
        double *tile = cur ? tile1 : tile0;
        if (!shared_row || i == L - 1) {
            cp_async_wait_all();
            __syncwarp();
            load_tile_row<NB>(e, tile, lane);
            if (!shared_row && i > 0) {                // prefetch the next row into the other buffer
                stage_row<NB>(cur ? tile0 : tile1, endp + (i - 1) * ers, lane);
                cp_async_commit();
                cur ^= 1;
            }
        }
        if (MASK && !((live >> j32) & 1u)) {           // masked row: nothing decoded, the symbol slot keeps what it held
            if (j32 == 0) {
                int64_t r = i + lane;
                if (r < L) sy[r] = (int16_t)my_sym;
            }
            continue;
        }
        RowTable<NB> T;
        build_row<NB>(e, __shfl_sync(FULL, mu_w, j32), __shfl_sync(FULL, sc_w, j32), mult, bits, lane, T);
        // ---- search: s = max{k : C[k] <= m}  (cifar_compress.py:60-61) -----------------------------
        uint32_t m = (uint32_t)ws.x & mask;
        int owner = 31 - __clz(__ballot_sync(FULL, T.base <= m));
        uint32_t acc = T.base, cs = T.base, ps = T.P[0];
        int js = 0;
#pragma unroll
        for (int j = 1; j < NB; ++j) {
            acc += T.P[j - 1];
            if (acc <= m) { cs = acc; ps = T.P[j]; js = j; }
        }
        cs = __shfl_sync(FULL, cs, owner);
        ps = __shfl_sync(FULL, ps, owner);
        int s = owner * NB + __shfl_sync(FULL, js, owner);
        if (lane == j32) my_sym = s;                                            // :62
        ws.decode(ps, cs, m, bits, lane);                                       // :63-65
        if (j32 == 0 || ws.err) {                      // block of rows done: coalesced symbol store
            int64_t r = (i & ~(int64_t)31) + lane;
            if (r < L && r >= i) sy[r] = (int16_t)my_sym;
            if (ws.err) break;
        }
    }
    cp_async_wait_all();
    ws.close(sv, b, lane);
}

template <int NB, bool MASK>
__global__ void __launch_bounds__(FW * 32) k_logistic_push(bsw_streams sv, int first, int count,
        const float *__restrict__ mu, int64_t mss, const float *__restrict__ sc, int64_t sss,
        const double *__restrict__ endp, int64_t ers, const int16_t *__restrict__ sym, int64_t L, int bits, int q,
        const uint32_t *__restrict__ rowmask) {
    extern __shared__ double smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int si = blockIdx.x * FW + warp;
    if (si >= count) return;
    int b = first + si;
    WarpStream ws;
    ws.open(sv, b);
    if (ws.err) return;
    ws.push_begin(lane);
    double *tile0 = smem + (size_t)warp * 2 * tile_doubles<NB>();
    double *tile1 = tile0 + tile_doubles<NB>();
    const float *mub = mu + (int64_t)si * mss, *scb = sc + (int64_t)si * sss;
    const int16_t *sy = sym + (int64_t)si * L;
    const double mult = (double)(((int64_t)1 << bits) - ((int64_t)1 << q));
    const bool shared_row = (ers == 0);
    const uint32_t *rm = MASK ? rowmask + (int64_t)si * (L >> 5) : nullptr;

    double e[NB];
    stage_row<NB>(tile0, endp, lane);
    cp_async_commit();
    float mu_w = 0.f, sc_w = 1.f;
    int sym_w = 0;
    uint32_t live = FULL;
    int cur = 0;
    for (int64_t i = 0; i < L; ++i) {
        int j32 = (int)(i & 31);
        if (j32 == 0) {
            int64_t r = i + lane;
            mu_w = r < L ? mub[r] : 0.f;
            sc_w = r < L ? scb[r] : 1.f;
            sym_w = r < L ? (int)sy[r] : 0;
            if (MASK) live = __ldg(rm + (i >> 5));
        }
        double *tile = cur ? tile1 : tile0;
        if (!shared_row || i == 0) {
            cp_async_wait_all();
            __syncwarp();
            load_tile_row<NB>(e, tile, lane);
            if (!shared_row && i + 1 < L) {
                stage_row<NB>(cur ? tile0 : tile1, endp + (i + 1) * ers, lane);
                cp_async_commit();
                cur ^= 1;
            }
        }
        if (MASK && !((live >> j32) & 1u)) continue;  // masked row: head and word stack untouched
        RowTable<NB> T;
        build_row<NB>(e, __shfl_sync(FULL, mu_w, j32), __shfl_sync(FULL, sc_w, j32), mult, bits, lane, T);
        int s = __shfl_sync(FULL, sym_w, j32);
        if ((unsigned)s >= (unsigned)(32 * NB)) { ws.err = BSW_E_INVALID; break; }    // reference: IndexError at self.pmfs[i, s]
        int owner = s / NB, js = s - owner * NB;
        uint32_t acc = T.base, cs = T.base, ps = T.P[0];
#pragma unroll
        for (int j = 1; j < NB; ++j) {
            acc += T.P[j - 1];
            if (j == js) { cs = acc; ps = T.P[j]; }
        }
        cs = __shfl_sync(FULL, cs, owner);
        ps = __shfl_sync(FULL, ps, owner);
        ws.encode(ps, cs, bits, lane);                                          // cifar_compress.py:50-54
        if (ws.err) break;
    }
    cp_async_wait_all();
    ws.push_end(lane);
    ws.close(sv, b, lane);
}

template <int NB>
static int launch_fused(bool push, bsw_streams *s, int first, int count, const float *mu, int64_t mss, const float *sc,
                        int64_t sss, const double *endp, int64_t ers, int16_t *sym, int64_t L, int bits, int q,
                        const uint32_t *rowmask, cudaStream_t st) {
    size_t smem = (size_t)FW * 2 * tile_doubles<NB>() * sizeof(double);
    const unsigned g = (count + FW - 1) / FW;
#define FUSED_LAUNCH(K)                                                                                                       \
    do {                                                                                                                      \
        BSW_CUDA(cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                            \
        K<<<g, FW * 32, smem, st>>>(*s, first, count, mu, mss, sc, sss, endp, ers, sym, L, bits, q, rowmask);                 \
    } while (0)
    if (push) {
        if (rowmask) FUSED_LAUNCH((k_logistic_push<NB, true>)); else FUSED_LAUNCH((k_logistic_push<NB, false>));
    } else {
        if (rowmask) FUSED_LAUNCH((k_logistic_pop<NB, true>)); else FUSED_LAUNCH((k_logistic_pop<NB, false>));
    }
#undef FUSED_LAUNCH
    BSW_LAUNCH_CHECK();
    return BSW_OK;
}
static int dispatch_fused(bool push, bsw_streams *s, int first, int count, const float *mu, int64_t mss, const float *sc,
                          int64_t sss, const double *endp, int64_t ers, int16_t *sym, int64_t L, int S, int bits, int q,
                          const uint32_t *rowmask, void *stream) {
    if (int rc = check_range(s, first, count)) return rc;
    BSW_REQUIRE(mu && sc && endp && sym && L > 0, "fused coder: null argument");
    BSW_REQUIRE(bits > 0 && bits <= 31 && q >= 0 && q < bits, "fused coder: bits/quantbits out of range");
    BSW_REQUIRE((ers == 0 || ers >= S) && (((uintptr_t)endp) & 7) == 0, "fused coder: endpoint rows must hold S doubles (+inf padded)");
    BSW_REQUIRE(!rowmask || (L & 31) == 0, "fused coder: a row mask needs a multiple of 32 rows");
    cudaStream_t st = (cudaStream_t)stream;
    switch (S) {
        case 32:   return launch_fused<1>(push, s, first, count, mu, mss, sc, sss, endp, ers, sym, L, bits, q, rowmask, st);
        case 64:   return launch_fused<2>(push, s, first, count, mu, mss, sc, sss, endp, ers, sym, L, bits, q, rowmask, st);
        case 128:  return launch_fused<4>(push, s, first, count, mu, mss, sc, sss, endp, ers, sym, L, bits, q, rowmask, st);
        case 256:  return launch_fused<8>(push, s, first, count, mu, mss, sc, sss, endp, ers, sym, L, bits, q, rowmask, st);
        case 512:  return launch_fused<16>(push, s, first, count, mu, mss, sc, sss, endp, ers, sym, L, bits, q, rowmask, st);
        case 1024: return launch_fused<32>(push, s, first, count, mu, mss, sc, sss, endp, ers, sym, L, bits, q, rowmask, st);
    }
    bsw_set_error("fused coder: support must be one of 32,64,...,1024 (got %d)", S);
    return BSW_E_INVALID;
}
extern "C" int bsw_logistic_push(bsw_streams *s, int first, int count, const float *mu, int64_t mss, const float *sc,
                                 int64_t sss, const double *endp, int64_t ers, const int16_t *sym, int64_t L, int S,
                                 int bits, int q, void *stream) {
    return dispatch_fused(true, s, first, count, mu, mss, sc, sss, endp, ers, (int16_t *)sym, L, S, bits, q, nullptr, stream);
}
extern "C" int bsw_logistic_pop(bsw_streams *s, int first, int count, const float *mu, int64_t mss, const float *sc,
                                int64_t sss, const double *endp, int64_t ers, int16_t *sym, int64_t L, int S, int bits,
                                int q, void *stream) {
    return dispatch_fused(false, s, first, count, mu, mss, sc, sss, endp, ers, sym, L, S, bits, q, nullptr, stream);
}
// The fused coder with a row mask (NULL = every row; L/32 words per stream, a clear bit (i & 31) of word i/32 skips row i):
// what the codec calls for the pixel level of a partial block.
int bsw_logistic_fused(bool pop, bsw_streams *s, int first, int count, const float *mu, int64_t mss, const float *sc,
                       int64_t sss, const double *endp, int64_t ers, int16_t *sym, int64_t L, int S, int bits, int q,
                       const uint32_t *rowmask, cudaStream_t st) {
    return dispatch_fused(!pop, s, first, count, mu, mss, sc, sss, endp, ers, sym, L, S, bits, q, rowmask, st);
}

// ================================================================================================
// Bin tables + centre gathers (a5, a6, a7 data)
// ================================================================================================
int bsw_rows6_build_meta(const double *endp, int64_t ers, int64_t L, int S, void *meta_dev, int *n_affine_host, cudaStream_t st);   // ans_rows6.cu
extern "C" int bsw_bins_create(bsw_bins **out, int nz, int zdim, int q, int xdim, const double *zend_host,
                               const double *zcen_host) {
    BSW_REQUIRE(out && nz > 0 && zdim > 0 && q > 0 && q <= 10 && zend_host && zcen_host, "bsw_bins_create: bad arguments");
    bsw_bins *b = new bsw_bins();
    b->nz = nz; b->zdim = zdim; b->q = q; b->S = 1 << q; b->xdim = xdim;
    const int S = b->S;
    // pad value of every endpoint row: any finite value this large gives cdf == 1.0 exactly in every kernel
    // (a literal +inf would turn the reciprocal-division shortcut into inf - inf)
    const double inf = 1e300;
    size_t rows = (size_t)nz * zdim;
    std::vector<double> pad(rows * S);
    for (size_t r = 0; r < rows; ++r) {
        memcpy(&pad[r * S], zend_host + r * (S - 1), sizeof(double) * (S - 1));
        pad[r * S + S - 1] = inf;
    }
    BSW_CUDA(cudaMalloc(&b->zend, sizeof(double) * rows * S));
    BSW_CUDA(cudaMalloc(&b->zcen, sizeof(double) * rows * S));
    BSW_CUDA(cudaMalloc(&b->xend, sizeof(double) * 256));
    BSW_CUDA(cudaMemcpy(b->zend, pad.data(), sizeof(double) * rows * S, cudaMemcpyHostToDevice));
    BSW_CUDA(cudaMemcpy(b->zcen, zcen_host, sizeof(double) * rows * S, cudaMemcpyHostToDevice));
    double xe[256];
    for (int k = 1; k <= 255; ++k) xe[k - 1] = (((double)k - 127.5) / 127.5) - 1. / 255.;   // rand.py:146-147
    xe[255] = inf;
    BSW_CUDA(cudaMemcpy(b->xend, xe, sizeof(xe), cudaMemcpyHostToDevice));
    // classify the rows once: levels whose rows are all uniform grids (every level discretize_kbins() builds,
    // discretization.py:105-118, and the pixel row) are coded by the affine-row kernels
    BSW_REQUIRE(nz <= 64, "bsw_bins_create: at most 64 levels");
    BSW_CUDA(cudaMalloc(&b->zmeta, (size_t)32 * rows));
    BSW_CUDA(cudaMalloc(&b->xmeta, 32));
    for (int l = 0; l < nz; ++l) {
        int n_aff = 0;
        b->zaffine[l] = 0;
        if (S >= 8) {
            if (int rc = bsw_rows6_build_meta(b->zend + (size_t)l * zdim * S, S, zdim, S, (uint8_t *)b->zmeta + (size_t)32 * l * zdim, &n_aff, nullptr)) return rc;
            b->zaffine[l] = n_aff == zdim;
        }
    }
    {
        int n_aff = 0;
        if (int rc = bsw_rows6_build_meta(b->xend, 0, 1, 256, b->xmeta, &n_aff, nullptr)) return rc;
        b->xaffine = n_aff == 1;
    }
    *out = b;
    return BSW_OK;
}
extern "C" int bsw_bins_level_is_uniform(const bsw_bins *b, int level) {
    if (!b) return 0;
    if (level < 0) return b->xaffine;
    return level < b->nz ? b->zaffine[level] : 0;
}
extern "C" int bsw_bins_destroy(bsw_bins *b) {
    if (!b) return BSW_OK;
    cudaFree(b->zend); cudaFree(b->zcen); cudaFree(b->xend); cudaFree(b->zmeta); cudaFree(b->xmeta);
    delete b;
    return BSW_OK;
}
extern "C" int bsw_bins_device_ptrs(bsw_bins *b, int level, const double **zend, const double **zcen, const double **xend) {
    BSW_REQUIRE(b && level >= 0 && level < b->nz, "bsw_bins_device_ptrs: level out of range");
    size_t off = (size_t)level * b->zdim * b->S;
    if (zend) *zend = b->zend + off;
    if (zcen) *zcen = b->zcen + off;
    if (xend) *xend = b->xend;
    return BSW_OK;
}

__global__ void k_gather_z(const double *__restrict__ cen, int zdim, int S, const int16_t *__restrict__ sym,
                           float *__restrict__ out, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int d = (int)(i % zdim);
    out[i] = (float)cen[(int64_t)d * S + sym[i]];           // cifar_compress.py:180,195 then .float() (cifar_train.py:392)
}
__global__ void k_gather_x(const uint8_t *__restrict__ x, float *__restrict__ out, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = (float)(((double)x[i] - 127.5) / 127.5);       // rand.py:151-152 centres, float64 -> float32
}
extern "C" int bsw_gather_zcentres(const bsw_bins *b, int level, const int16_t *sym, float *out, int64_t n_streams, void *stream) {
    BSW_REQUIRE(b && level >= 0 && level < b->nz && sym && out && n_streams > 0, "bsw_gather_zcentres: bad arguments");
    int64_t n = n_streams * b->zdim;
    k_gather_z<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(b->zcen + (size_t)level * b->zdim * b->S, b->zdim, b->S, sym, out, n);
    BSW_LAUNCH_CHECK();
    return BSW_OK;
}
extern "C" int bsw_gather_xcentres(const uint8_t *x, float *out, int64_t n, void *stream) {
    BSW_REQUIRE(x && out && n > 0, "bsw_gather_xcentres: bad arguments");
    k_gather_x<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, out, n);
    BSW_LAUNCH_CHECK();
    return BSW_OK;
}
