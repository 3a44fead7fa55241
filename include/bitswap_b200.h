/*
 * bitswap_b200.h -- C ABI of the B200-native Bit-Swap hot path.
 *
 * The reference (fhkingma/bitswap @ dfe0bf7d) is pure Python and has no FFI: its
 * "plugin interface" for this path is a handful of Python call signatures
 * (SURVEY.md 8b).  Each entry point below names the reference call it replaces.
 * Python binds these with ctypes (bitswap_b200/_lib.py); INTEGRATION.md shows the
 * stub a maintainer of the reference would add to cifar_compress.py.
 *
 * Conventions
 *   - every function returns a bsw_status (0 = ok); nothing throws across the ABI
 *   - "dev" pointers are CUDA device pointers owned by the caller (e.g. torch
 *     tensors); the library never frees them.  "host" pointers are ordinary memory.
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream); every
 *     kernel is enqueued on it, no call synchronises unless it says so.
 *   - an ANS stream == one reference state list: 32-bit words bottom-first plus a
 *     64-bit head (cifar_compress.py:157-159).  B streams = B independent chains.
 */
#ifndef BITSWAP_B200_H
#define BITSWAP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    BSW_OK          = 0,
    BSW_E_UNDERFLOW = 1,   /* reference: IndexError from x.pop(-2)          (cifar_compress.py:65)    */
    BSW_E_OVERFLOW  = 2,   /* word stack capacity exhausted (reference lists grow without bound)      */
    BSW_E_BADTABLE  = 3,   /* reference: AssertionError on the cdf table    (cifar_compress.py:45-46) */
    BSW_E_INVALID   = 4,   /* bad argument                                                            */
    BSW_E_CUDA      = 5    /* CUDA runtime error; see bsw_last_error()                                */
} bsw_status;

const char *bsw_last_error(void);
int         bsw_version(void);
/* 1 if this build contains the tcgen05 conv path (bsw_model_desc.use_tensor_cores may be set). */
int         bsw_has_tensor_cores(void);
/* Measures this GPU's peak float64 FMA rate (DFMA/s, lanes) with a register-resident kernel: the roofline
 * denominator of the float64 row-table kernel (the driver's MEASURED_PEAKS.json has no FP64 figure). */
int         bsw_measure_fp64_peak(double *dfma_per_s);
/* Device self-test: the lean cdf of the throughput kernels vs the exact (IEEE division + libdevice exp) cdf on n
 * random finite (endpoint, mu, sigma) triples, far tails included.  example_host: 5 doubles or NULL. */
int         bsw_selftest_cdf(int64_t n, uint64_t seed, int64_t *mismatches_host, double *example_host);
/* worst |screening cdf - exact cdf| over n random arguments, in units of 2^-51 (the screening window is 64 units) */
int         bsw_selftest_cdf_apx(int64_t n, uint64_t seed, double *worst_units_host);

/* ------------------------------------------------------------------------------------------------
 * Stream sets: B device-resident ANS states.
 * Replaces: the Python list `state` (cifar_compress.py:157-159) -- create/import == building the
 * list, export == reading it back / pickle.dump (cifar_compress.py:265-266).
 * ---------------------------------------------------------------------------------------------- */
typedef struct bsw_streams bsw_streams;
typedef struct bsw_bins bsw_bins;

/* capacity_words is rounded up to a multiple of 32. */
int bsw_streams_create(bsw_streams **out, int n_streams, int64_t capacity_words);
int bsw_streams_destroy(bsw_streams *s);
int bsw_streams_count(const bsw_streams *s);
int64_t bsw_streams_capacity(const bsw_streams *s);

/* Host import: stream (first+i) receives words_host[offsets[i] .. offsets[i+1]) and heads_host[i].
 * Synchronous. */
int bsw_streams_import(bsw_streams *s, int first, int count, const uint32_t *words_host,
                       const int64_t *offsets_host, const uint64_t *heads_host);
/* Every stream receives the same words/head (the reference seeds every experiment identically,
 * cifar_compress.py:93,157).  Synchronous. */
int bsw_streams_fill(bsw_streams *s, const uint32_t *words_host, int64_t nwords, uint64_t head);
/* Word counts (list length - 1), heads and per-stream status flags (bsw_status values). Synchronous. */
int bsw_streams_sizes(bsw_streams *s, int64_t *nwords_host, uint64_t *heads_host, int32_t *flags_host);
/* Lowest word count each stream has reached since import/fill: the part of the initial random words that was never
 * borrowed and can be trimmed from a stored bitstream (demo_compress.py:137,160 `excess_state_len`). Synchronous. */
int bsw_streams_min_words(bsw_streams *s, int64_t *min_host);
/* Word count of each stream right after the FIRST pop of its chain since import/fill (-1: none yet): the reference's
 * len(restbits) - 1, from which it reports `totalbits` and the cumulative moving average (cifar_compress.py:190-192,254,259).
 * Recorded by bsw_codec_encode.  Synchronous. */
int bsw_streams_rest_words(bsw_streams *s, int64_t *rest_host);
/* Packed export: stream i's words go to words_host[offsets_host[i] ...). Synchronous. */
int bsw_streams_export(bsw_streams *s, int first, int count, uint32_t *words_host, const int64_t *offsets_host);
/* Device-side packed (de)serialisation, async on `stream`: all streams' words gathered into one contiguous device
 * buffer (capacity >= total words; offsets_dev holds count+1 int64 prefix sums, heads_dev count uint64), or scattered back
 * (unpack requires every stream's length <= capacity; it also resets flags).  A host export is then three memcpys. */
int bsw_streams_pack(bsw_streams *s, int first, int count, uint32_t *words_dev, int64_t *offsets_dev, uint64_t *heads_dev,
                     void *stream);
int bsw_streams_unpack(bsw_streams *s, int first, int count, const uint32_t *words_dev, const int64_t *offsets_dev,
                       const uint64_t *heads_dev, void *stream);
/* Trimmed forms: only words[base_b .. n_b) of every stream travel, base_b = the lowest depth the stack ever reached
 * (bsw_streams_min_words) -- the initial random words below it were never borrowed and the receiver re-creates them from
 * the seed (demo_compress.py:137,160; demo_decompress.py:176-186).  base_dev: int32 [count], written by pack, read by
 * unpack.  unpack_trimmed writes above base_b into streams that already hold the initial words (bsw_streams_fill /
 * import), and flags BSW_E_OVERFLOW instead of writing past a stream's capacity. */
int bsw_streams_pack_trimmed(bsw_streams *s, int first, int count, uint32_t *words_dev, int64_t *offsets_dev,
                             uint64_t *heads_dev, int32_t *base_dev, void *stream);
int bsw_streams_unpack_trimmed(bsw_streams *s, int first, int count, const uint32_t *words_dev, const int64_t *offsets_dev,
                               const uint64_t *heads_dev, const int32_t *base_dev, void *stream);
/* Raw device views for device-resident pipelines (NCCL gathers, custom kernels). */
int bsw_streams_device_ptrs(bsw_streams *s, uint32_t **words_dev, int32_t **nwords_dev, uint64_t **heads_dev,
                            int32_t **flags_dev);
/* Device-side: sum over streams of (nwords) -> *total_dev (int64), async on `stream`. */
int bsw_streams_total_words(bsw_streams *s, int64_t *total_dev, void *stream);

/* ------------------------------------------------------------------------------------------------
 * a1  ANS.__init__ (cifar_compress.py:13-46): float64 pmfs [L,S] -> integer tables.
 *     P_dev [L,S] uint32, C_dev [L,S+1] uint32 (C[:,S] == 2^bits).  err_dev (int32, may be NULL) is
 *     set to BSW_E_BADTABLE if a row fails the reference's assertions.
 * ---------------------------------------------------------------------------------------------- */
int bsw_ans_tables(const double *pmfs_dev, int64_t L, int S, int bits, int quantbits,
                   uint32_t *P_dev, uint32_t *C_dev, int32_t *err_dev, void *stream);

/* ------------------------------------------------------------------------------------------------
 * a2/a3  ANS.encode / ANS.decode (cifar_compress.py:48-67) over given integer tables, batched over
 *     the set's streams [first, first+count).  Tables: P [.,L,S], C [.,L,S+1]; table_stream_stride
 *     = elements between consecutive streams' tables (0: one table shared by all streams).
 *     Symbols: int32 [count, L].  push walks rows ascending, pop descending, exactly as the
 *     reference loops do.
 * ---------------------------------------------------------------------------------------------- */
int bsw_ans_push(bsw_streams *s, int first, int count, const uint32_t *P_dev, const uint32_t *C_dev,
                 int64_t P_stream_stride, int64_t C_stream_stride, const int32_t *sym_dev,
                 int64_t L, int S, int bits, void *stream);
int bsw_ans_pop(bsw_streams *s, int first, int count, const uint32_t *P_dev, const uint32_t *C_dev,
                int64_t P_stream_stride, int64_t C_stream_stride, int32_t *sym_dev,
                int64_t L, int S, int bits, void *stream);

/* ------------------------------------------------------------------------------------------------
 * a4  logistic_cdf + pmf assembly (utils/torch/rand.py:67-68, cifar_compress.py:182-184).
 *     endpoints_dev: row r starts at endpoints_dev + r*endp_row_stride and holds S-1 doubles
 *     (stride 0 = one row shared by all, as ImageBins' identical rows allow).
 *     mu/scale: double, indexed [r*ms] (ms = 0 broadcasts, as the prior does at :245).
 *     Writes pmfs_dev [L,S] float64 -- the debug/export path of the parity ladder (P2); the hot
 *     path never materialises pmfs.
 * ---------------------------------------------------------------------------------------------- */
int bsw_logistic_pmfs(const double *endpoints_dev, int64_t endp_row_stride, const double *mu_dev,
                      const double *scale_dev, int64_t ms, int64_t L, int S, double *pmfs_dev, void *stream);

/* a4+a1 fused, materialised: integer tables straight from (endpoints, mu, scale).  Used for tables
 * that are shared by every stream (the Logistic(0,1) prior, cifar_compress.py:245-247). */
int bsw_logistic_tables(const double *endpoints_dev, int64_t endp_row_stride, const double *mu_dev,
                        const double *scale_dev, int64_t ms, int64_t L, int S, int bits, int quantbits,
                        uint32_t *P_dev, uint32_t *C_dev, void *stream);

/* ------------------------------------------------------------------------------------------------
 * a4+a1+a2 / a4+a1+a3 fused hot kernels: one warp per stream builds each row's table in registers
 * (float64 logistic cdf -> trunc -> remnant at the row argmax -> scan) and codes the symbol; tables
 * never reach HBM.  Replaces the per-level sequence
 *     cdfs = logistic_cdf(...); pmfs = ...; ANS(pmfs, bits, q).encode/decode(state, ...)
 * of cifar_compress.py:182-187,197-202.
 *     mu_dev/scale_dev: float32 (the nets' outputs, up-cast to float64 in the kernel as
 *     model/cifar_train.py:375-376 does); element [b*mu_stream_stride + r].  A stream stride of 0
 *     shares the vector between streams (the unconditional x-scale, cifar_train.py:411).
 *     endpoints as above but each row holds S doubles, the last one +inf (library layout, see
 *     bsw_bins_*).  S must be a multiple of 32 and <= 1024.
 *     sym: int16 [count, L].
 * ---------------------------------------------------------------------------------------------- */
int bsw_logistic_push(bsw_streams *s, int first, int count, const float *mu_dev, int64_t mu_stream_stride,
                      const float *scale_dev, int64_t scale_stream_stride, const double *endpoints_dev,
                      int64_t endp_row_stride, const int16_t *sym_dev, int64_t L, int S, int bits,
                      int quantbits, void *stream);
int bsw_logistic_pop(bsw_streams *s, int first, int count, const float *mu_dev, int64_t mu_stream_stride,
                     const float *scale_dev, int64_t scale_stream_stride, const double *endpoints_dev,
                     int64_t endp_row_stride, int16_t *sym_dev, int64_t L, int S, int bits,
                     int quantbits, void *stream);

/* Two-phase variants (the throughput path of the codec): a fully parallel float64 row-table kernel followed by the
 * serial integer coder; same arguments and bit-identical results, plus caller-provided 16-byte aligned device scratch
 * of at least bsw_logistic_scratch_bytes(count, L, S, 0) bytes (the last argument is ignored; kept for ABI stability).
 * Two kernel families: the generic one (any sorted endpoint rows) and the affine-row one for rows that are uniform
 * grids -- which is every row discretize_kbins() builds (discretization.py:105-118) and the ImageBins pixel row
 * (utils/torch/rand.py:146-147).  These two entry points probe the rows on every call (one small kernel + a stream
 * synchronise); the codec uses the classification bsw_bins_create made. */
int64_t bsw_logistic_scratch_bytes(int count, int64_t L, int S, int full_tables);
/* Kernel family for bsw_logistic_*_2p and the codec: -1 = by row classification (default; BSW_ROWS_MODE overrides),
 * 0 = generic kernels only, 1 = affine-row kernels for every row (non-uniform rows take the exact path per bin). */
int bsw_set_rows_mode(int mode);
/* 1 if every endpoint row of `level` (or the pixel row, level = -1) is a uniform grid. */
int bsw_bins_level_is_uniform(const bsw_bins *b, int level);
/* Debug: with verify on, every affine-row table launch also evaluates the exact function for every bin.
 * bsw_rows6_verify_read returns and resets {bins that differ from the exact function (must be 0), worst error of a
 * trusted bin in thousandths of its window, bins checked, bins that took the exact path}. */
int bsw_rows6_set_verify(int on);
/* Mapping of the affine-row table kernel: lanes of a warp that share one row (2, 4, 8 or 32; 0 = default 4, i.e. eight
 * rows per warp).  Every setting emits the same integers; exposed for A/B timing and the parity test. */
int bsw_rows6_set_lanes_per_row(int lpr);
/* Launch shape of the tcgen05 convolutions, a bit mask: 8 / 16 = dense 3x3 / dense 5x5 on the pair-tile kernel (2-CTA
 * clusters issuing cta_group::2 M = 256, N = 256 MMAs, one image per pair, weight tile split across the pair), 1 / 2 / 4 =
 * dense 3x3 / dense 5x5 / in-convs on the persistent kernel (one CTA per SM walking half-image tiles with a TMEM
 * ping-pong); a clear bit = one CTA per tile.  -1 = default (BSW_TC_PERSIST if set, else 24).  Bit-identical results. */
int bsw_set_conv_mode(int mode);
int bsw_rows6_verify_read(uint64_t *out4_host);
int bsw_logistic_push_2p(bsw_streams *s, int first, int count, const float *mu_dev, int64_t mu_stream_stride,
                         const float *scale_dev, int64_t scale_stream_stride, const double *endpoints_dev,
                         int64_t endp_row_stride, const int16_t *sym_dev, int64_t L, int S, int bits, int quantbits,
                         void *scratch_dev, int64_t scratch_bytes, void *stream);
int bsw_logistic_pop_2p(bsw_streams *s, int first, int count, const float *mu_dev, int64_t mu_stream_stride,
                        const float *scale_dev, int64_t scale_stream_stride, const double *endpoints_dev,
                        int64_t endp_row_stride, int16_t *sym_dev, int64_t L, int S, int bits, int quantbits,
                        void *scratch_dev, int64_t scratch_bytes, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Bin tables on the device.
 * Replaces: the tensors returned by discretize() (discretization.py:9-99) and ImageBins
 * (utils/torch/rand.py:134-153); the library keeps its own padded copy (each endpoint row padded
 * with +1e300 to S entries so that cdf_{S-1} == 1 falls out of the same formula).
 * ---------------------------------------------------------------------------------------------- */
/* zendpoints_host [nz, zdim, S-1], zcentres_host [nz, zdim, S] float64 (reference layout). */
int bsw_bins_create(bsw_bins **out, int nz, int zdim, int quantbits, int xdim,
                    const double *zendpoints_host, const double *zcentres_host);
int bsw_bins_destroy(bsw_bins *b);
/* Device views: padded z endpoints of a level [zdim, S]; z centres of a level [zdim, S]; the single
 * padded x endpoint row [256]. */
int bsw_bins_device_ptrs(bsw_bins *b, int level, const double **zend_dev, const double **zcen_dev,
                         const double **xend_dev);

/* a5  centre gathers (cifar_compress.py:180,195): symbols -> float32 values fed to the nets
 *     (float64 table value cast to float32, model/cifar_train.py:324,392).
 *     z: out[b,d] = (float) zcentres[level, d, sym[b,d]];  x: out[b,d] = (float)((x-127.5)/127.5). */
int bsw_gather_zcentres(const bsw_bins *b, int level, const int16_t *sym_dev, float *out_dev, int64_t n_streams,
                        void *stream);
int bsw_gather_xcentres(const uint8_t *x_dev, float *out_dev, int64_t n, void *stream);

/* ------------------------------------------------------------------------------------------------
 * f3  Sampling epilogue and bin fit of discretize() (discretization.py:30-118).
 * minmax_dev: uint32 [2 * dim] running extrema (order-preserving encoding), reset before a level.
 * bsw_discretize_sample: out[r,d] = float16(mu[r,d] + scale[r,d] * eps), eps = log(u) - log1p(-u) with u clamped to
 *   [bound, 1 - bound] (utils/torch/rand.py:6-20), and folds the float16 values into the extrema.  scale_row_stride 0 = one
 *   shared scale row.  bsw_discretize_fold: fold float16 samples produced elsewhere (the top-level prior draw).
 * bsw_discretize_edges: np.linspace(min, max, 2^q + 1) per dimension -> endpoints [dim][2^q - 1] and centres [dim][2^q]
 *   in float64 (KBinsDiscretizer strategy='uniform', discretization.py:105-118).
 * ---------------------------------------------------------------------------------------------- */
int bsw_discretize_reset(uint32_t *minmax_dev, int dim, void *stream);
int bsw_discretize_sample(const float *mu_dev, const float *scale_dev, int64_t scale_row_stride, const float *u_dev, float bound,
                          void *out_half_dev, uint32_t *minmax_dev, int64_t rows, int dim, void *stream);
int bsw_discretize_fold(const void *samples_half_dev, uint32_t *minmax_dev, int64_t rows, int dim, void *stream);
int bsw_discretize_edges(const uint32_t *minmax_dev, int dim, int quantbits, double *endpoints_dev, int64_t endp_row_stride,
                         double *centres_dev, int64_t cen_row_stride, void *stream);

/* ------------------------------------------------------------------------------------------------
 * a8-a10  The inference-time VAE.
 * Replaces: Model.infer(i)(given) / Model.generate(i)(given) in compressing mode
 * (model/cifar_train.py:315-438; imagenetcrop_train.py:306-315,417) and the WnConv2d / ResNetLayer /
 * Squeeze2d / UnSqueeze2d forwards they run (utils/torch/modules.py:98-106,175-241).
 * ---------------------------------------------------------------------------------------------- */
typedef struct bsw_model bsw_model;
typedef struct {
    int32_t xc;            /* image channels C (xs = (C,32,32)) */
    int32_t nz;
    int32_t zchannels;
    int32_t nprocessing;
    int32_t kernel_size;   /* 3 */
    int32_t resdepth;
    int32_t reswidth;
    int32_t cond_xscale;   /* imagenetcrop: x-scale from a conv head */
    int32_t max_batch;     /* activations are preallocated for this many images */
    int32_t use_tensor_cores; /* 1: tcgen05 path for the W->W convs (needs padded width 256); 0: fp32 SIMT */
} bsw_model_desc;

int bsw_model_create(bsw_model **out, const bsw_model_desc *desc);
int bsw_model_destroy(bsw_model *m);
/* Loads one WnConv2d by its reference state_dict prefix (e.g. "infer_res0.0.res252layer1.conv1"):
 * v [O,I,k,k], gain [O], b [O] float32 host arrays.  Weight normalisation
 * w = v * g/(||v||+1e-10), g = softplus(gain) if loggain else gain (modules.py:98-105) is folded here,
 * once.  Synchronous. */
int bsw_model_load_conv(bsw_model *m, const char *prefix, const float *v_host, const float *gain_host,
                        const float *b_host, int O, int I, int k, int loggain);
/* The unconditional x-scale parameter gen_std [C,32,32] (model/cifar_train.py:306-308). */
int bsw_model_load_gen_std(bsw_model *m, const float *gen_std_host);
/* Call after all tensors are loaded; checks completeness. */
int bsw_model_finalize(bsw_model *m);

/* given_dev float32 [n, dim_in] flat CHW (what `given.float()` is in the reference);
 * mu_dev/scale_dev float32 [n, dim_out] flat CHW.  For generate(0) without cond_xscale the scale does
 * not depend on the input: scale_dev receives the [xdim] vector replicated n times only if
 * scale_per_stream != 0, else one [xdim] row. */
int bsw_vae_infer(bsw_model *m, int level, const float *given_dev, int64_t n, float *mu_dev, float *scale_dev,
                  void *stream);
int bsw_vae_generate(bsw_model *m, int level, const float *given_dev, int64_t n, float *mu_dev, float *scale_dev,
                     int scale_per_stream, void *stream);

/* ------------------------------------------------------------------------------------------------
 * a11/a12  The Bit-Swap recursion, device resident.
 * Replaces: the sender loop body of cifar_compress.py:175-204,244-250 and the receiver loop body of
 * :283-317 for `count` streams at once (one image per stream per call; chain images by calling again).
 * x_dev uint8 [count, C,32,32].  No host round trip between levels; errors land in the per-stream
 * flags (bsw_streams_sizes).  `scheme`: 0 = Bit-Swap, 1 = BB-ANS (cifar_compress.py:205-242,319-352).
 * ---------------------------------------------------------------------------------------------- */
typedef struct bsw_codec bsw_codec;
int bsw_codec_create(bsw_codec **out, bsw_model *m, bsw_bins *b, int max_batch);
int bsw_codec_destroy(bsw_codec *c);
int bsw_codec_encode(bsw_codec *c, bsw_streams *s, int first, int count, const uint8_t *x_dev, int scheme,
                     void *stream);
int bsw_codec_decode(bsw_codec *c, bsw_streams *s, int first, int count, uint8_t *x_dev, int scheme,
                     void *stream);
/* Partial blocks (the edges of an image that is not a multiple of 32 on a side).  extent_dev int32 [count, 2] =
 * (valid_rows, valid_cols) of each stream's block, each in [1, 32]; pixel (c, y, x) is valid iff y < valid_rows and
 * x < valid_cols.  Masked pixels are not coded: both sides overwrite them with the edge-replicate fill
 * x[c][min(y, valid_rows-1)][min(x, valid_cols-1)] before infer(0) sees the block, the x-level push/pop skip their rows,
 * and decode returns the fill there.  The latent levels are coded as for a whole block.  An extent outside [1, 32] flags
 * that stream BSW_E_INVALID; the other streams are unaffected.  extent_dev == NULL is exactly bsw_codec_encode/decode,
 * and all-(32, 32) extents give bit-identical streams. */
int bsw_codec_encode_ext(bsw_codec *c, bsw_streams *s, int first, int count, const uint8_t *x_dev,
                         const int32_t *extent_dev, int scheme, void *stream);
int bsw_codec_decode_ext(bsw_codec *c, bsw_streams *s, int first, int count, uint8_t *x_dev,
                         const int32_t *extent_dev, int scheme, void *stream);
/* Number of kernel launches the last encode/decode call enqueued (bench.py's gpu_launches). */
int64_t bsw_codec_last_launches(const bsw_codec *c);
/* Stream placement inside one encode/decode call: 0 (default) = every kernel on the caller's stream; 1 = conv kernels
 * on a high-priority internal stream, coder kernels on a low-priority one, chained with events and joined back into
 * `stream` at the end (an experiment in co-scheduling tensor-bound and FP64-bound CTAs; measured no gain on B200). */
int bsw_codec_set_dual_stream(bsw_codec *c, int on);
/* Coder variant: 1 (default) = two-phase (ans_rows.cu: fully parallel float64 row tables, then the serial integer
 * coder), 0 = fused one-warp-per-stream kernels (bsw_logistic_push/pop).  Bit-identical results. */
int bsw_codec_set_two_phase(bsw_codec *c, int on);
/* Per-kernel-category device time (CUDA events on the launching stream) accumulated since profiling was
 * enabled.  ms_out/n_out: 12 entries {misc, conv_in, conv_dense3x3, conv_dense5x5, conv_head, pop_z, push_z,
 * pop_x, push_x, prior, rows_z, rows_x} (rows_* = phase A of the two-phase coder; pop/push = phase B).  enable: 1 = reset and start, 0 = reset and stop, -1 = read only.  Synchronises. */
int bsw_codec_profile(bsw_codec *c, int enable, double *ms_out, int64_t *n_out);

#ifdef __cplusplus
}
#endif
#endif /* BITSWAP_B200_H */
