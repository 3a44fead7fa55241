// The bits-back recursions, device resident (sm_100a).
//
// Reference being replaced (fhkingma/bitswap @ dfe0bf7d):
//   Bit-Swap sender   cifar_compress.py:175-204, 244-250      receiver  :283-317
//   BB-ANS  sender    cifar_compress.py:205-242, 244-250      receiver  :319-352
// One call codes ONE image per stream for `count` streams.  Every step is a kernel enqueued on the
// caller's stream; symbols, centres, mu/sigma and the ANS state stay in HBM between levels -- the
// reference's 2*nz GPU<->CPU round trips per image (cifar_compress.py:42-43,66) do not exist here.
#include <stdlib.h>
#include <vector>
#include "bsw_common.cuh"
#include "nets.cuh"

struct bsw_codec {
    bsw_model *m;
    bsw_bins *b;
    int max_batch, nz, zdim, xdim, q, S;
    float *given, *mu, *scale;          // [max_batch, max(xdim, zdim)]
    float *mu2, *scale2;                // second mu/sigma pair: in overlap mode infer() and generate() results are alive at once
    int16_t *sym[2];                    // ping-pong latent symbols [max_batch, zdim]
    int16_t *xsym;                      // [max_batch, xdim] pixels as int16 symbols
    uint32_t *rowmask;                  // [max_batch, xdim / 32] pixel rows a partial block codes (bsw_codec_encode_ext)
    std::vector<int16_t *> zs;          // BB-ANS: all nz latents
    void *scratch;                      // two-phase coder: pairs / coarse cdf of one level
    size_t scratch_bytes;
    void *scratch_push = nullptr;       // overlap mode: the push side's (P_s, C_s, M) rows get their own buffer
    size_t scratch_push_bytes = 0;
    int two_phase;                      // 1: ans_rows.cu path (default), 0: fused one-warp-per-stream kernels
    uint32_t *priorP, *priorC;
    uint32_t *priorCoarse = nullptr;    // prior cdf at every 32nd bin + dummy fix: lets the prior pop use k_pop_full
    uint2 *priorFix = nullptr;          // Logistic(0,1) prior tables over zendpoints[-1], shared by all streams
    int64_t launches;
    BswProf prof;
    // overlap mode (bsw_codec_set_dual_stream(c, 1)): the recursion is enqueued as a DAG on three internal streams --
    // st_conv (nets), st_rows (parallel float64 table kernels), st_ser (serial integer coder kernels) -- see the comment
    // above bsw_codec_encode.
    cudaStream_t st_conv = nullptr, st_rows = nullptr, st_ser = nullptr;
    cudaEvent_t ev[16];
    int ev_next = 0;
    int dual_stream = 0;
};

// internal int16-symbol variants of the table-driven coder (ans_kernels.cu)
int bsw_ans_push_i16(bsw_streams *s, int first, int count, const uint32_t *P, const uint32_t *C, int64_t pss, int64_t css,
                     const int16_t *sym, int64_t L, int S, int bits, cudaStream_t st);
int bsw_ans_pop_i16(bsw_streams *s, int first, int count, const uint32_t *P, const uint32_t *C, int64_t pss, int64_t css,
                    int16_t *sym, int64_t L, int S, int bits, cudaStream_t st);

size_t bsw_rows_scratch_bytes(int count, int64_t L);
int bsw_streams_mark_rest(bsw_streams *s, int first, int count, cudaStream_t st);
int bsw_rows_mode();
int bsw_prior_coarse(const uint32_t *C, int64_t L, int S, uint32_t *coarse, uint2 *fix, cudaStream_t st);
int bsw_pop_shared_table(bsw_streams *s, int first, int count, const uint32_t *P, const uint32_t *coarse, const uint2 *fix,
                         int16_t *sym, int64_t L, int S, int bits, cudaStream_t st);
int bsw_logistic_2p(int phase, bool pop, bsw_streams *s, int first, int count, const float *mu, int64_t mss, const float *sc,
                    int64_t sss, const double *endp, int64_t ers, const void *meta, int16_t *sym, int64_t L, int S, int bits, int q,
                    void *scratch, size_t scratch_bytes, const uint32_t *rowmask, cudaStream_t st);
int bsw_logistic_fused(bool pop, bsw_streams *s, int first, int count, const float *mu, int64_t mss, const float *sc,
                       int64_t sss, const double *endp, int64_t ers, int16_t *sym, int64_t L, int S, int bits, int q,
                       const uint32_t *rowmask, cudaStream_t st);

__global__ void k_u8_to_i16(const uint8_t *__restrict__ in, int16_t *__restrict__ out, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[i];
}
__global__ void k_i16_to_u8(const int16_t *__restrict__ in, uint8_t *__restrict__ out, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (uint8_t)in[i];
}

// ---- partial blocks: extents [count][2] = (valid_rows, valid_cols) of each stream's 32x32 block, each in [1, 32] ----------
// Pixel p of a CHW block (c = p >> 10, y = (p >> 5) & 31, x = p & 31) is valid iff y < valid_rows && x < valid_cols.  The
// masked pixels are not coded; they hold the edge-replicate fill x[c][min(y, vr-1)][min(x, vc-1)] on both sides, so that
// the inference net sees the same block when the encoder reads it and when the decoder rebuilds it.
__device__ __forceinline__ int ext_clamp(int v) { return v < 1 ? 1 : (v > 32 ? 32 : v); }
// position the fill copies pixel p from (p itself when it is valid); out-of-range extents are clamped here only to keep
// the read in bounds -- k_rowmask has already flagged that stream, and no coder kernel touches it again
__device__ __forceinline__ int fill_src(int p, int vr, int vc) {
    const int y = (p >> 5) & 31, x = p & 31;
    return (p & ~1023) | (min(y, ext_clamp(vr) - 1) << 5) | min(x, ext_clamp(vc) - 1);
}
// One word per (stream, channel, image row): word k of a stream holds the 32 pixels of row k & 31 of channel k >> 5, i.e.
// exactly the pixel-level rows [32k, 32k + 32) the serial coder kernels walk.  An extent outside [1, 32] flags the stream
// BSW_E_INVALID (the first failure of a stream is the one kept) and every later coder kernel skips it.
__global__ void k_rowmask(const int32_t *__restrict__ ext, int64_t n, int wps, uint32_t *__restrict__ mask,
                          int32_t *__restrict__ flags) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int si = (int)(i / wps), k = (int)(i - (int64_t)si * wps);
    const int vr = ext[2 * si], vc = ext[2 * si + 1];
    const bool ok = vr >= 1 && vr <= 32 && vc >= 1 && vc <= 32;
    mask[i] = (ok && (k & 31) < vr) ? (vc == 32 ? 0xffffffffu : (1u << vc) - 1u) : 0u;
    if (!ok && k == 0 && flags[si] == BSW_OK) flags[si] = BSW_E_INVALID;
}
// encode: uint8 -> int16 symbols with the fill applied on the way
__global__ void k_u8_to_i16_fill(const uint8_t *__restrict__ in, int16_t *__restrict__ out, int64_t n, int xdim,
                                 const int32_t *__restrict__ ext) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int si = (int)(i / xdim), p = (int)(i - (int64_t)si * xdim);
    out[i] = in[(int64_t)si * xdim + fill_src(p, ext[2 * si], ext[2 * si + 1])];
}
// decode: the fill in place on the popped symbols -- reads valid positions only, writes masked positions only
__global__ void k_fill_x(int16_t *__restrict__ x, int64_t n, int xdim, const int32_t *__restrict__ ext) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int si = (int)(i / xdim), p = (int)(i - (int64_t)si * xdim);
    const int src = fill_src(p, ext[2 * si], ext[2 * si + 1]);
    if (src != p) x[i] = x[(int64_t)si * xdim + src];
}

extern "C" int bsw_codec_create(bsw_codec **out, bsw_model *m, bsw_bins *b, int max_batch) {
    BSW_REQUIRE(out && m && b && max_batch >= 1, "bsw_codec_create: bad arguments");
    BSW_REQUIRE(m->finalized, "bsw_codec_create: model not finalized");
    BSW_REQUIRE(b->nz == m->d.nz && b->zdim == m->zdim, "bsw_codec_create: bins do not match the model");
    BSW_REQUIRE(max_batch <= m->d.max_batch, "bsw_codec_create: max_batch exceeds the model's");
    bsw_codec *c = new bsw_codec();
    c->m = m; c->b = b; c->max_batch = max_batch;
    c->nz = b->nz; c->zdim = b->zdim; c->xdim = m->xdim; c->q = b->q; c->S = b->S;
    size_t dim = (size_t)(c->xdim > c->zdim ? c->xdim : c->zdim);
    BSW_CUDA(cudaMalloc(&c->given, sizeof(float) * dim * max_batch));
    BSW_CUDA(cudaMalloc(&c->mu, sizeof(float) * dim * max_batch));
    BSW_CUDA(cudaMalloc(&c->scale, sizeof(float) * dim * max_batch));
    BSW_CUDA(cudaMalloc(&c->mu2, sizeof(float) * dim * max_batch));
    BSW_CUDA(cudaMalloc(&c->scale2, sizeof(float) * dim * max_batch));
    BSW_CUDA(cudaMalloc(&c->sym[0], sizeof(int16_t) * c->zdim * max_batch));
    BSW_CUDA(cudaMalloc(&c->sym[1], sizeof(int16_t) * c->zdim * max_batch));
    BSW_CUDA(cudaMalloc(&c->xsym, sizeof(int16_t) * c->xdim * max_batch));
    BSW_CUDA(cudaMalloc(&c->rowmask, sizeof(uint32_t) * (c->xdim / 32) * max_batch));
    // symbol buffers start as valid symbols (0): a stream that is skipped because of its error flag leaves them as they
    // are, and the centre gathers index tables with them
    BSW_CUDA(cudaMemset(c->sym[0], 0, sizeof(int16_t) * c->zdim * max_batch));
    BSW_CUDA(cudaMemset(c->sym[1], 0, sizeof(int16_t) * c->zdim * max_batch));
    BSW_CUDA(cudaMemset(c->xsym, 0, sizeof(int16_t) * c->xdim * max_batch));
    c->zs.assign(c->nz, nullptr);
    {
        size_t a = bsw_rows_scratch_bytes(max_batch, c->zdim), b2 = bsw_rows_scratch_bytes(max_batch, c->xdim);
        c->scratch_bytes = a > b2 ? a : b2;
        BSW_CUDA(cudaMalloc(&c->scratch, c->scratch_bytes));
        c->scratch_push_bytes = (size_t)max_batch * dim * 16;
        BSW_CUDA(cudaMalloc(&c->scratch_push, c->scratch_push_bytes));
        c->two_phase = 1;
    }
    // prior tables: Logistic(0,1) over the top level's endpoints, identical for every stream and image
    // (cifar_compress.py:245-247) -> built once, with the same float64 kernel math as every other table.
    BSW_CUDA(cudaMalloc(&c->priorP, sizeof(uint32_t) * (size_t)c->zdim * c->S));
    BSW_CUDA(cudaMalloc(&c->priorC, sizeof(uint32_t) * (size_t)c->zdim * (c->S + 1)));
    double ms[2] = {0.0, 1.0}, *dms = nullptr;
    BSW_CUDA(cudaMalloc(&dms, sizeof(ms)));
    BSW_CUDA(cudaMemcpy(dms, ms, sizeof(ms), cudaMemcpyHostToDevice));
    const double *zend = b->zend + (size_t)(c->nz - 1) * c->zdim * c->S;
    int rc = bsw_logistic_tables(zend, c->S, dms, dms + 1, 0, c->zdim, c->S, 31, c->q, c->priorP, c->priorC, nullptr);
    if (!rc && c->S >= 128) {
        BSW_CUDA(cudaMalloc(&c->priorCoarse, sizeof(uint32_t) * (size_t)c->zdim * (c->S / 32)));
        BSW_CUDA(cudaMalloc(&c->priorFix, sizeof(uint2) * (size_t)c->zdim));
        rc = bsw_prior_coarse(c->priorC, c->zdim, c->S, c->priorCoarse, c->priorFix, nullptr);
    }
    BSW_CUDA(cudaDeviceSynchronize());
    cudaFree(dms);
    if (rc) return rc;
    c->launches = 0;
    int lo_p = 0, hi_p = 0;
    BSW_CUDA(cudaDeviceGetStreamPriorityRange(&lo_p, &hi_p));          // (numerically lower = higher priority)
    // equal priorities: on this part a running higher-priority kernel keeps lower-priority CTAs from being dispatched at
    // all (measured: convs on a high-priority stream and table kernels on a low-priority one took the SUM of their solo
    // times), so priorities can only serialise
    (void)hi_p;
    BSW_CUDA(cudaStreamCreateWithPriority(&c->st_ser, cudaStreamNonBlocking, lo_p));
    BSW_CUDA(cudaStreamCreateWithPriority(&c->st_conv, cudaStreamNonBlocking, lo_p));
    BSW_CUDA(cudaStreamCreateWithPriority(&c->st_rows, cudaStreamNonBlocking, lo_p));
    for (auto &e : c->ev) BSW_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    *out = c;
    return BSW_OK;
}

extern "C" int bsw_codec_destroy(bsw_codec *c) {
    if (!c) return BSW_OK;
    cudaFree(c->given); cudaFree(c->mu); cudaFree(c->scale); cudaFree(c->mu2); cudaFree(c->scale2); cudaFree(c->scratch_push);
    cudaFree(c->sym[0]); cudaFree(c->sym[1]); cudaFree(c->xsym); cudaFree(c->rowmask);
    for (auto p : c->zs) cudaFree(p);
    cudaFree(c->priorP); cudaFree(c->priorC); cudaFree(c->scratch); cudaFree(c->priorCoarse); cudaFree(c->priorFix);
    for (cudaStream_t st : {c->st_conv, c->st_rows, c->st_ser}) if (st) cudaStreamDestroy(st);
    for (auto &e : c->ev) cudaEventDestroy(e);
    delete c;
    return BSW_OK;
}
extern "C" int64_t bsw_codec_last_launches(const bsw_codec *c) { return c ? c->launches : 0; }

/* 1: overlap mode -- nets, table kernels and serial coder kernels on three internal streams, chained by events as the
 *    dependency graph allows (see bsw_codec_encode); 0 (default): everything in program order on the caller's stream. */
extern "C" int bsw_codec_set_dual_stream(bsw_codec *c, int on) {
    BSW_REQUIRE(c, "null codec");
    c->dual_stream = on > 0 ? 1 : 0;
    return BSW_OK;
}

extern "C" int bsw_codec_set_two_phase(bsw_codec *c, int on) {
    BSW_REQUIRE(c, "null codec");
    c->two_phase = on ? 1 : 0;
    return BSW_OK;
}

// Per-category kernel timing for bench.py's roofline (CUDA events on the launching stream).
extern "C" int bsw_codec_profile(bsw_codec *c, int enable, double *ms_out, int64_t *n_out) {
    BSW_REQUIRE(c, "null codec");
    c->prof.collect();
    if (ms_out) for (int i = 0; i < CAT_COUNT; ++i) ms_out[i] = c->prof.ms[i];
    if (n_out) for (int i = 0; i < CAT_COUNT; ++i) n_out[i] = c->prof.n[i];
    if (enable >= 0) { c->prof.reset(); c->prof.on = enable != 0; }
    return BSW_OK;
}

#define RC(call) do { if (int rc_ = (call)) return rc_; } while (0)

namespace {
// One encode/decode call.  Three stream roles -- conv (nets + the gathers that feed them), rows (phase A: parallel float64
// table kernels) and ser (phase B: the serial integer coder, the only kernels that touch the ANS state).  In the default
// mode all three are the caller's stream and hop() is a no-op: plain program order.  In overlap mode they are the codec's
// internal streams and hop(a, b) makes everything enqueued on a so far happen-before what follows on b.
struct Ctx {
    bsw_codec *c; bsw_streams *s; int first, count;
    cudaStream_t conv, rows, ser;
    cudaStream_t caller = nullptr;
    int nl = 0;
    const int32_t *ext = nullptr;       // partial blocks: extents [count][2] on the device (NULL: whole blocks)
    const uint32_t *xmask = nullptr;    // ... and the pixel-level row mask built from them
    void begin(cudaStream_t user) {
        caller = user;
        if (c->dual_stream) {
            conv = c->st_conv; rows = c->st_rows; ser = c->st_ser;
            cudaEvent_t e = next_event();
            cudaEventRecord(e, user);
            for (cudaStream_t t : {conv, rows, ser}) cudaStreamWaitEvent(t, e, 0);
        } else conv = rows = ser = user;
    }
    void end() {
        if (!c->dual_stream) return;
        for (cudaStream_t t : {conv, rows, ser}) hop(t, caller);
    }
    cudaEvent_t next_event() {
        cudaEvent_t e = c->ev[c->ev_next];
        c->ev_next = (c->ev_next + 1) & 15;
        return e;
    }
    void hop(cudaStream_t from, cudaStream_t to) {
        if (from == to) return;
        cudaEvent_t e = next_event();        // (a wait captures the record that precedes it, so the small pool can be reused)
        cudaEventRecord(e, from);
        cudaStreamWaitEvent(to, e, 0);
    }
    const double *zend(int lvl) const { return c->b->zend + (size_t)lvl * c->zdim * c->S; }
    // row metadata of a level whose rows are all uniform grids (-> affine-row kernels), else NULL (-> generic kernels)
    const void *zmeta(int lvl) const {
        return (c->b->zaffine[lvl] && bsw_rows_mode() != 0) ? (const uint8_t *)c->b->zmeta + (size_t)32 * lvl * c->zdim : nullptr;
    }
    const void *xmeta() const { return (c->b->xaffine && bsw_rows_mode() != 0) ? c->b->xmeta : nullptr; }
    // mu/sigma of the inference nets live in (mu, scale), those of the generative nets in (mu2, scale2)
    float *mu_of(bool infer) const { return infer ? c->mu : c->mu2; }
    float *sc_of(bool infer) const { return infer ? c->scale : c->scale2; }
    int net(bool infer, int zi) {
        return bsw_model_run(c->m, infer, zi, c->given, count, mu_of(infer), sc_of(infer), infer ? 1 : 0, conv, &nl, &c->prof);
    }
    int gather_x(const uint8_t *x) {
        ++nl;
        c->prof.begin(CAT_MISC, conv);
        int rc = bsw_gather_xcentres(x, c->given, (int64_t)count * c->xdim, conv);
        c->prof.end(conv);
        return rc;
    }
    int gather_x16(const int16_t *x);
    // net input of infer(0) on the encode side: the pixels as given, or for partial blocks the filled symbols
    int gather_x_in(const uint8_t *x) {
        if (!ext) return gather_x(x);
        hop(rows, conv);                                  // (the fill is enqueued on the rows stream)
        return gather_x16(c->xsym);
    }
    // the row mask of the pixel level, on `st` (the stream of the first coder kernel that reads the flags it sets)
    int build_mask(cudaStream_t st) {
        const int wps = c->xdim / 32;
        const int64_t n = (int64_t)count * wps;
        k_rowmask<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(ext, n, wps, c->rowmask, s->flags + first);
        BSW_LAUNCH_CHECK();
        ++nl;
        xmask = c->rowmask;
        return BSW_OK;
    }
    // decode: the fill on the popped pixel symbols, on the serial stream right after the pop (the hop ser -> conv that
    // follows the pop orders it before the gather that reads them)
    int fill_x() {
        if (!ext) return BSW_OK;
        const int64_t n = (int64_t)count * c->xdim;
        k_fill_x<<<(unsigned)((n + 255) / 256), 256, 0, ser>>>(c->xsym, n, c->xdim, ext);
        BSW_LAUNCH_CHECK();
        ++nl;
        return BSW_OK;
    }
    int gather_z(int lvl, const int16_t *sym) {
        ++nl;
        c->prof.begin(CAT_MISC, conv);
        int rc = bsw_gather_zcentres(c->b, lvl, sym, c->given, count, conv);
        c->prof.end(conv);
        return rc;
    }
    // One logistic table level, pop or push, from the nets' (mu, sigma) of `from_infer`.  L = zdim over level `lvl`
    // endpoints (lvl >= 0) or the pixel level (lvl = -1: ImageBins endpoints, one shared row, 8-bit quantisation,
    // cifar_compress.py:202).  The caller has already ordered `rows` after the net that produced mu/sigma.
    int level(bool pop, int lvl, bool from_infer, int16_t *sym) {
        const bool x = lvl < 0;
        const int64_t L = x ? c->xdim : c->zdim;
        const int S = x ? 256 : c->S, q = x ? 8 : c->q;
        const double *endp = x ? c->b->xend : zend(lvl);
        const int64_t ers = x ? 0 : c->S;
        const void *meta = x ? xmeta() : zmeta(lvl);
        const float *mu = mu_of(from_infer), *sc = sc_of(from_infer);
        const int64_t sss = x ? (c->m->d.cond_xscale ? c->xdim : 0) : c->zdim;
        const int cat_rows = x ? CAT_ROWS_X : CAT_ROWS_Z;
        const int cat_ser = x ? (pop ? CAT_POP_X : CAT_PUSH_X) : (pop ? CAT_POP_Z : CAT_PUSH_Z);
        const uint32_t *rm = x ? xmask : nullptr;
        if (!c->two_phase) {
            hop(rows, ser);
            ++nl;
            c->prof.begin(cat_ser, ser);
            int rc = bsw_logistic_fused(pop, s, first, count, mu, L, sc, sss, endp, ers, sym, L, S, 31, q, rm, ser);
            c->prof.end(ser);
            return rc;
        }
        // the push side has its own scratch in overlap mode: the next level's pop tables may be built while the serial
        // push of this level still reads its rows
        void *scr = (!pop && c->dual_stream) ? c->scratch_push : c->scratch;
        const size_t scr_bytes = (!pop && c->dual_stream) ? c->scratch_push_bytes : c->scratch_bytes;
        nl += 2;
        c->prof.begin(cat_rows, rows);
        int rc = bsw_logistic_2p(0, pop, s, first, count, mu, L, sc, sss, endp, ers, meta, sym, L, S, 31, q, scr, scr_bytes, rm, rows);
        c->prof.end(rows);
        if (rc) return rc;
        hop(rows, ser);
        c->prof.begin(cat_ser, ser);
        rc = bsw_logistic_2p(1, pop, s, first, count, mu, L, sc, sss, endp, ers, meta, sym, L, S, 31, q, scr, scr_bytes, rm, ser);
        c->prof.end(ser);
        return rc;
    }
    int push_prior(const int16_t *sym) {
        ++nl;
        c->prof.begin(CAT_PRIOR, ser);
        int rc = bsw_ans_push_i16(s, first, count, c->priorP, c->priorC, 0, 0, sym, c->zdim, c->S, 31, ser);
        c->prof.end(ser);
        return rc;
    }
    int pop_prior(int16_t *sym) {
        ++nl;
        c->prof.begin(CAT_PRIOR, ser);
        int rc = c->priorCoarse
            ? bsw_pop_shared_table(s, first, count, c->priorP, c->priorCoarse, c->priorFix, sym, c->zdim, c->S, 31, ser)
            : bsw_ans_pop_i16(s, first, count, c->priorP, c->priorC, 0, 0, sym, c->zdim, c->S, 31, ser);
        c->prof.end(ser);
        return rc;
    }
};
__global__ void k_gather_x16(const int16_t *__restrict__ x, float *__restrict__ out, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (float)(((double)x[i] - 127.5) / 127.5);
}
int Ctx::gather_x16(const int16_t *x) {
    ++nl;
    int64_t n = (int64_t)count * c->xdim;
    k_gather_x16<<<(unsigned)((n + 255) / 256), 256, 0, conv>>>(x, c->given, n);
    BSW_LAUNCH_CHECK();
    return BSW_OK;
}
}  // namespace

static int codec_args_ok(bsw_codec *c, bsw_streams *s, int first, int count, const void *x) {
    BSW_REQUIRE(c && s && x, "bsw_codec: null argument");
    BSW_REQUIRE(first >= 0 && count >= 1 && first + count <= s->B, "bsw_codec: stream range out of bounds");
    BSW_REQUIRE(count <= c->max_batch, "bsw_codec: count exceeds the codec's max_batch");
    return BSW_OK;
}
static int ensure_zs(bsw_codec *c) {
    for (auto &p : c->zs)
        if (!p) {
            BSW_CUDA(cudaMalloc(&p, sizeof(int16_t) * c->zdim * c->max_batch));
            BSW_CUDA(cudaMemset(p, 0, sizeof(int16_t) * c->zdim * c->max_batch));
        }
    return BSW_OK;
}
static int codec_ext_ok(bsw_codec *c, const int32_t *ext) {
    BSW_REQUIRE(!ext || c->xdim % 1024 == 0, "bsw_codec: extents need 32x32 pixel blocks");
    return BSW_OK;
}

// Dependencies of one Bit-Swap sender level (receiver: the same with the roles of the nets swapped):
//     infer(zi)  ->  tables q(z_zi)  ->  POP z_zi  ->  generate(zi)  ->  tables p(z_zi-1 | z_zi)  ->  PUSH z_zi-1
//                                            \->  infer(zi+1)  ->  tables q(z_zi+1)  ->  POP z_zi+1 (after PUSH z_zi-1)
// Only the serial coder kernels touch the ANS state, and only they are ordered by it; infer(zi+1) needs the popped
// symbols, not the push.  In overlap mode the conv stream therefore runs  ... generate(zi), infer(zi+1), generate(zi+1) ...
// back to back while the float64 table kernels of the push run beside infer(zi+1) on the rows stream: tensor-pipe work
// and FP64-pipe work of ONE chain share the SMs (the persistent conv kernel leaves room for a table CTA on every SM).
// Buffers that make this legal: separate (mu, sigma) for the two nets, separate scratch for the push rows.
// extent (may be NULL): partial blocks, see k_rowmask.  The masked pixels are overwritten by the fill before infer(0) sees
// the block, and the x-level push codes only the valid rows.
extern "C" int bsw_codec_encode_ext(bsw_codec *c, bsw_streams *s, int first, int count, const uint8_t *x, const int32_t *extent,
                                    int scheme, void *stream) {
    RC(codec_args_ok(c, s, first, count, x));
    RC(codec_ext_ok(c, extent));
    Ctx k{c, s, first, count};
    k.ext = extent;
    k.begin((cudaStream_t)stream);
    const int nz = c->nz;
    int64_t nx = (int64_t)count * c->xdim;
    if (extent) {
        RC(k.build_mask(k.rows));                        // (the hop rows -> ser before the first pop orders it)
        k_u8_to_i16_fill<<<(unsigned)((nx + 255) / 256), 256, 0, k.rows>>>(x, c->xsym, nx, c->xdim, extent);
    } else {
        k_u8_to_i16<<<(unsigned)((nx + 255) / 256), 256, 0, k.rows>>>(x, c->xsym, nx);   // (read by the push_x table kernel)
    }
    BSW_LAUNCH_CHECK();
    ++k.nl;
    int16_t *zsym = c->sym[0], *ztop = c->sym[1];
    if (scheme == 0) {
        // Bit-Swap sender (cifar_compress.py:178-204)
        for (int zi = 0; zi < nz; ++zi) {
            if (zi == 0) RC(k.gather_x_in(x)); else RC(k.gather_z(zi - 1, zsym));        // :180
            RC(k.net(true, zi));                                                            // :181
            k.hop(k.conv, k.rows);
            RC(k.level(true, zi, true, ztop));                                              // :182-187
            if (zi == 0) { RC(bsw_streams_mark_rest(s, first, count, k.ser)); ++k.nl; }     // :190-192 restbits (first pop of a chain only)
            k.hop(k.ser, k.conv);
            RC(k.gather_z(zi, ztop));                                                       // :195
            RC(k.net(false, zi));                                                           // :196
            k.hop(k.conv, k.rows);
            RC(k.level(false, zi == 0 ? -1 : zi - 1, false, zi == 0 ? c->xsym : zsym));    // :197-202
            int16_t *t = zsym; zsym = ztop; ztop = t;                                       // :204
        }
    } else {
        // BB-ANS sender (cifar_compress.py:208-242): all pops first, then all pushes
        RC(ensure_zs(c));
        for (int zi = 0; zi < nz; ++zi) {
            if (zi == 0) RC(k.gather_x_in(x)); else RC(k.gather_z(zi - 1, c->zs[zi - 1]));
            RC(k.net(true, zi));
            k.hop(k.conv, k.rows);
            RC(k.level(true, zi, true, c->zs[zi]));
            if (zi == 0) { RC(bsw_streams_mark_rest(s, first, count, k.ser)); ++k.nl; }     // :224-226 restbits
            k.hop(k.ser, k.conv);
        }
        for (int zi = 0; zi < nz; ++zi) {
            RC(k.gather_z(zi, c->zs[zi]));
            RC(k.net(false, zi));
            k.hop(k.conv, k.rows);
            RC(k.level(false, zi == 0 ? -1 : zi - 1, false, zi == 0 ? c->xsym : c->zs[zi - 1]));
            k.hop(k.ser, k.conv);                    // (mu2/sigma2 and the push scratch are rewritten by the next level)
        }
        zsym = c->zs[nz - 1];
    }
    RC(k.push_prior(zsym));                                                                 // :245-250
    k.end();
    c->launches = k.nl;
    return BSW_OK;
}
extern "C" int bsw_codec_encode(bsw_codec *c, bsw_streams *s, int first, int count, const uint8_t *x, int scheme, void *stream) {
    return bsw_codec_encode_ext(c, s, first, count, x, nullptr, scheme, stream);
}

// extent (may be NULL): partial blocks.  The x-level pop decodes only the valid rows; right after it the fill rebuilds the
// masked pixels, so infer(0) sees the encoder's block and the returned block holds the fill there.
extern "C" int bsw_codec_decode_ext(bsw_codec *c, bsw_streams *s, int first, int count, uint8_t *x, const int32_t *extent,
                                    int scheme, void *stream) {
    RC(codec_args_ok(c, s, first, count, x));
    RC(codec_ext_ok(c, extent));
    Ctx k{c, s, first, count};
    k.ext = extent;
    k.begin((cudaStream_t)stream);
    if (extent) RC(k.build_mask(k.ser));
    const int nz = c->nz;
    int16_t *ztop = c->sym[0], *sym = c->sym[1];
    if (scheme == 0) {
        // Bit-Swap receiver (cifar_compress.py:283-317)
        RC(k.pop_prior(ztop));                                                              // :284-289
        k.hop(k.ser, k.conv);
        for (int zi = nz - 1; zi >= 0; --zi) {
            RC(k.gather_z(zi, ztop));                                                       // :296
            RC(k.net(false, zi));                                                           // :297
            k.hop(k.conv, k.rows);
            RC(k.level(true, zi == 0 ? -1 : zi - 1, false, zi == 0 ? c->xsym : sym));       // :298-303
            if (zi == 0) RC(k.fill_x());
            k.hop(k.ser, k.conv);
            if (zi == 0) RC(k.gather_x16(c->xsym)); else RC(k.gather_z(zi - 1, sym));       // :306
            RC(k.net(true, zi));                                                            // :307
            k.hop(k.conv, k.rows);
            RC(k.level(false, zi, true, ztop));                                             // :308-313
            int16_t *t = ztop; ztop = sym; sym = t;                                         // :315
        }
    } else {
        // BB-ANS receiver (cifar_compress.py:319-352)
        RC(ensure_zs(c));
        RC(k.pop_prior(c->zs[nz - 1]));
        k.hop(k.ser, k.conv);
        for (int zi = nz - 1; zi >= 0; --zi) {
            RC(k.gather_z(zi, c->zs[zi]));
            RC(k.net(false, zi));
            k.hop(k.conv, k.rows);
            RC(k.level(true, zi == 0 ? -1 : zi - 1, false, zi == 0 ? c->xsym : c->zs[zi - 1]));
            if (zi == 0) RC(k.fill_x());
            k.hop(k.ser, k.conv);
        }
        for (int zi = nz - 1; zi >= 0; --zi) {
            if (zi == 0) RC(k.gather_x16(c->xsym)); else RC(k.gather_z(zi - 1, c->zs[zi - 1]));
            RC(k.net(true, zi));
            k.hop(k.conv, k.rows);
            RC(k.level(false, zi, true, c->zs[zi]));
            k.hop(k.ser, k.conv);                    // (mu/sigma and the push scratch are rewritten by the next level)
        }
    }
    int64_t nx = (int64_t)count * c->xdim;
    k_i16_to_u8<<<(unsigned)((nx + 255) / 256), 256, 0, k.ser>>>(c->xsym, x, nx);
    BSW_LAUNCH_CHECK();
    k.end();
    c->launches = k.nl + 1;
    return BSW_OK;
}
extern "C" int bsw_codec_decode(bsw_codec *c, bsw_streams *s, int first, int count, uint8_t *x, int scheme, void *stream) {
    return bsw_codec_decode_ext(c, s, first, count, x, nullptr, scheme, stream);
}
