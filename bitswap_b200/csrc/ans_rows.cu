// Two-phase logistic coder (sm_100a): the throughput path of the device-resident codec.
//
// The fused kernels of ans_kernels.cu keep one warp per stream busy with the whole row table, which leaves
// the FP64 pipe 27 % utilised at 1024 streams (profiles/r1_ncu_logistic_pop_v1.md: 7 warps per SM, long
// dependent DFMA chains).  The table of a row does not depend on the ANS head, only the *search* does, so:
//
//   phase A  (k_rows_push / k_rows_pop)   one warp per (stream,row), fully parallel over count x L rows:
//            float64 logistic cdf -> trunc -> remnant at the row argmax (ANS.__init__ semantics,
//            cifar_compress.py:28-39).  Streaming reductions only, so few registers and high occupancy.
//            push: emits the (P_s, C_s) pair of the symbol being coded            ->  8 B per row
//            pop : emits the integer cdf at every 32nd bin ("coarse cdf", 32 x 4 B) and (argmax, remnant)
//   phase B  (k_push_pairs / k_pop_coarse) one warp per stream, serial in the head as the reference is
//            (cifar_compress.py:48-67): push consumes the pairs; pop finds the 32-bin chunk containing
//            m = head & mask in the coarse cdf, recomputes just that chunk's 33 cdf values with the same
//            float64 function (bit-identical by construction) and finishes the search with a warp scan.
//
// Results are bit-identical to the fused kernels (integer sums are associative; the cdf function is shared).
#include <stdlib.h>
#include <type_traits>
#include <string.h>
#include "bsw_common.cuh"

#define FULL 0xffffffffu

namespace {

struct WarpStream2 {          // same state handling as ans_kernels.cu's WarpStream
    uint32_t *words;
    uint64_t x;
    int len, cap, wbase, err;
    uint32_t wbuf;
    __device__ __forceinline__ void open(const bsw_streams &sv, int b) {
        words = sv.words + (int64_t)b * sv.cap; x = sv.heads[b]; len = sv.nwords[b]; cap = (int)sv.cap;
        err = sv.flags[b]; wbase = -1; wbuf = 0;
    }
    __device__ __forceinline__ void close(const bsw_streams &sv, int b, int lane) {
        if (lane == 0) { sv.heads[b] = x; sv.nwords[b] = len; sv.flags[b] = err; if (len < sv.minwords[b]) sv.minwords[b] = len; }
    }
    __device__ __forceinline__ uint32_t pop_word(int lane) {
        int idx = len - 1;
        if (wbase < 0 || idx < wbase) { wbase = idx & ~31; wbuf = words[wbase + lane]; }
        len = idx;
        return __shfl_sync(FULL, wbuf, idx - wbase);
    }
    __device__ __forceinline__ void push_begin(int lane) {
        wbase = len & ~31;
        wbuf = (wbase + lane < len) ? words[wbase + lane] : 0u;
    }
    __device__ __forceinline__ void push_word(uint32_t w, int lane) {
        if (lane == len - wbase) wbuf = w;
        ++len;
        if (len - wbase == 32) { words[wbase + lane] = wbuf; wbase += 32; }
    }
    __device__ __forceinline__ void push_end(int lane) { if (lane < len - wbase) words[wbase + lane] = wbuf; }
    __device__ __forceinline__ void encode(uint32_t p, uint32_t c, int bits, int lane) {      // cifar_compress.py:51-54
        uint64_t lim = ((((uint64_t)1 << 32) >> bits) << 32) * (uint64_t)p;
        if (x >= lim) {
            if (len >= cap) { err = BSW_E_OVERFLOW; return; }
            push_word((uint32_t)x, lane);
            x >>= 32;
        }
        uint64_t qd = x / p;
        x = (qd << bits) + (x - qd * p) + c;
    }
    // same recurrence with the division replaced by a multiply with M = floor((2^64-1)/p) computed in the parallel phase:
    // floor(x*M / 2^64) is floor(x/p) or one less, so a single correction makes it exact
    __device__ __forceinline__ void encode_magic(uint32_t p, uint32_t c, uint64_t M, int bits, int lane) {
        uint64_t lim = ((((uint64_t)1 << 32) >> bits) << 32) * (uint64_t)p;
        if (x >= lim) {
            if (len >= cap) { err = BSW_E_OVERFLOW; return; }
            push_word((uint32_t)x, lane);
            x >>= 32;
        }
        uint64_t qd = __umul64hi(x, M);
        uint64_t rm = x - qd * p;
        if (rm >= p) { rm -= p; ++qd; }
        x = (qd << bits) + rm + c;
    }
    __device__ __forceinline__ void decode(uint32_t p, uint32_t c, uint32_t m, int bits, int lane) {   // :63-65
        x = (uint64_t)p * (x >> bits) + m - c;
        if (x < ((uint64_t)1 << 32)) {
            if (len <= 0) { err = BSW_E_UNDERFLOW; return; }
            x = (x << 32) | pop_word(lane);
        }
    }
};

constexpr int RW = 16;       // warps per CTA in phase A: 512 threads x <=64 registers = half an SM's register file, so two
                             // of these CTAs fill an SM, or one of them sits beside one k_conv_tc CTA (codec.cu overlap)

// ---- phase A ----------------------------------------------------------------------------------------------------
// One CTA = one row index for RW (=16) streams, one warp per stream.  The row's endpoints (shared by every stream) are
// staged once per CTA into a padded shared-memory tile; lane l then owns the NB consecutive bins [l*NB, l*NB+NB), so the
// cdf of the previous bin is already in a register (one shuffle per row instead of two per bin) and the 32-bin chunk
// totals the pop side needs are lane-local sums (no per-chunk warp reduction).  ~42 issued instructions per cdf value,
// 27 of them on the FP64 pipe.
// Tile layout: lane l's NB endpoints are contiguous and start at double index l*(NB+1): odd stride, conflict-free for the
// lane-blocked 8-byte reads.
template <int NB>
struct RowTile {
    static constexpr int STRIDE = NB + 1;
    static constexpr int DOUBLES = 32 * STRIDE;
};

__device__ __forceinline__ uint32_t smem_u32r(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// exact integer pmf (before the +1) of bin j of this lane's block: the rare path of the screened kernel
template <int NB, int STRIDE>
__device__ __noinline__ uint32_t rows_exact_pm(const double *tile, int lane, int j0, int t, double m, double s, double rs, double mult) {
    const int j = j0 + t;                                 // (added here so that the hot loop does not carry j0+1..j0+3)
    const double c = bsw_cdf_fast(tile[lane * STRIDE + j], m, s, rs);
    double p = 0.0;                                       // lower edge of bin 0 is cdf = 0 (cifar_compress.py:184)
    if (j > 0) p = bsw_cdf_fast(tile[lane * STRIDE + j - 1], m, s, rs);
    else if (lane > 0) p = bsw_cdf_fast(tile[(lane - 1) * STRIDE + NB - 1], m, s, rs);
    return __double2uint_rz(__dmul_rn(__dsub_rn(c, p), mult));
}

// APX = true (default): every cdf value comes from the 15-instruction screening function bsw_cdf_apx; the pmf is formed
// in 2^-20 fixed point with one FMA against a 2^52-type magic constant, and any bin whose scaled pmf lands within
// BSW_APX_WINDOW of an integer boundary (about 1.2e-4 of them) is recomputed with the exact bsw_cdf_fast.  The integers
// this kernel emits are therefore those of the exact function, which is what k_pop_coarse re-evaluates and what the
// fused kernels produce.  APX = false (BSW_ROWS_EXACT=1) evaluates the exact function for every bin.
template <int NB, bool POP, bool APX>
__global__ void __launch_bounds__(RW * 32, 2) k_rows(int count, int64_t L, const float *__restrict__ mu, int64_t mss,
        const float *__restrict__ sc, int64_t sss, const double *__restrict__ endp, int64_t ers,
        const int16_t *__restrict__ sym, int bits, int q, uint4 *__restrict__ pairs, uint32_t *__restrict__ coarse,
        uint2 *__restrict__ fix, const BswApxRegs KA) {
    constexpr int S = 32 * NB;
    using RT = RowTile<NB>;
    __shared__ __align__(16) double tile[RT::DOUBLES];
    __shared__ __align__(16) double t32[APX ? BSW_APX_TABLE_DOUBLES : 2];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t row = blockIdx.x;                      // row index i within the level
    const int si = blockIdx.y * RW + warp;               // stream
    const double *e = endp + row * ers;
    if (APX) bsw_apx_table_fill(t32, threadIdx.x, RW * 32);
    for (int k = threadIdx.x; k < S; k += RW * 32) tile[(k / NB) * RT::STRIDE + (k % NB)] = __ldg(e + k);
    __syncthreads();
    if (si >= count) return;
    const double m = (double)mu[(int64_t)si * mss + row], s = (double)sc[(int64_t)si * sss + row];
    const double rs = __ddiv_rn(1.0, s);
    const double mult = (double)(((int64_t)1 << bits) - ((int64_t)1 << q));
    const double mult2 = mult * 1048576.0;               // pmf in 2^-20 fixed point: < 2^51 for bits <= 31
    const double magic2 = 6755399441055744.0 + (double)BSW_APX_WINDOW;
    int sy = 0;
    if (!POP) sy = (int)sym[(int64_t)si * L + row];
    const int owner = sy / NB, js = sy - owner * NB;     // push: lane and in-lane position of the coded symbol

    BswExpRegs K;
    if (!APX) K.load();
    const double *my = tile + lane * RT::STRIDE;
    const uint32_t tl = smem_u32r(t32) + 8u * lane;
    // The screening cdf needs |t| <= 690 (its exponent arithmetic has no range checks).  Rows are sorted, so if both ends
    // of the row are inside that range for this stream's (mu, sigma) every bin is, and the three clamp instructions per
    // value are skipped (warp-uniform: a warp is one stream).  Needle-sharp x rows take the clamped loop.
    bool wide = true;
    if (APX && S > 2) {
        const double t_lo = __dmul_rn(__dsub_rn(tile[0], m), rs);
        const double t_hi = __dmul_rn(__dsub_rn(tile[((S - 2) / NB) * RT::STRIDE + ((S - 2) % NB)], m), rs);
        wide = !(fabs(t_lo) <= 690.0 && fabs(t_hi) <= 690.0);
    }
    auto cdf_at = [&](int j, auto clampc) -> double {
        if (APX) return bsw_cdf_apx<decltype(clampc)::value>(my[j], m, rs, tl, KA);
        return bsw_cdf_fast_regs(my[j], m, s, rs, K);
    };
    // cdf at my last endpoint first: the next lane needs it as the lower neighbour of its first bin.  The row's very
    // last entry is the +1e300 pad: t clamps to +690 and the cdf comes out as exactly 1.0, the reference's
    // `1. - cdfs[:,-1]` upper bound of the last bin (cifar_compress.py:184).
    const double c_last = cdf_at(NB - 1, std::true_type{});
    const double up = __shfl_up_sync(FULL, c_last, 1);
    double prev = lane == 0 ? 0.0 : up;
    constexpr int G = NB >= 4 ? 4 : NB;                  // bins per group
    // running state of my block: sum, the group holding the (first) maximum, and for push the integer cdf below the symbol
    uint32_t lsum = 0, lbest = 0, pre = 0, pv = 0;
    uint32_t bestv[G];
    int bestj0 = 0;
#pragma unroll
    for (int t = 0; t < G; ++t) bestv[t] = 0;
    auto group = [&](int j0, auto last_group, auto clampc) {
        uint32_t vv[G];
        bool doubt[G];
        bool any = false;
        uint32_t all_hi = 0x80000000u;
#pragma unroll
        for (int t = 0; t < G; ++t) {
            const double c = (decltype(last_group)::value && t == G - 1) ? c_last : cdf_at(j0 + t, clampc);
            if (APX) {
                // z = 1.5*2^52 + WINDOW + pmf*2^20: the mantissa of z holds the fixed-point pmf, shifted by WINDOW so that
                // "low 20 bits < 2*WINDOW" means "within WINDOW of a truncation boundary".  The funnel shift drops the low
                // 20 bits; what remains is the integer pmf with the 2^51 magic bit on top (bit 31).
                const double z = __fma_rn(__dsub_rn(c, prev), mult2, magic2);
                const uint32_t raw = __funnelshift_r((uint32_t)__double2loint(z), (uint32_t)__double2hiint(z), 20);
                // a pmf that truncates to 0 needs no second look: the exact value then lies in (-1, 1) as well
                doubt[t] = ((uint32_t)__double2loint(z) & (0xfffffu & ~(2u * BSW_APX_WINDOW - 1u))) == 0u && raw != 0x80000000u;
                any |= doubt[t];
                all_hi &= raw;                            // bit 31 clear = negative pmf (unsorted endpoints): exact path
                vv[t] = raw + 0x80000001u;                                                 // :29 trunc, :32 +1
            } else {
                vv[t] = __double2uint_rz(__dmul_rn(__dsub_rn(c, prev), mult)) + 1u;
            }
            prev = c;
        }
        if (APX && (any || !(all_hi & 0x80000000u))) {
            const bool all = !(all_hi & 0x80000000u);
#pragma unroll
            for (int t = 0; t < G; ++t)
                if (doubt[t] || all) vv[t] = rows_exact_pm<NB, RT::STRIDE>(tile, lane, j0, t, m, s, rs, mult) + 1u;
        }
        uint32_t gsum = 0, gmax = 0;
#pragma unroll
        for (int t = 0; t < G; ++t) { gsum += vv[t]; gmax = max(gmax, vv[t]); }
        lsum += gsum;
        if (gmax > lbest) {                               // strict: the earlier group keeps a tie (:35 first maximum)
            lbest = gmax; bestj0 = j0;
#pragma unroll
            for (int t = 0; t < G; ++t) bestv[t] = vv[t];
        }
        if (!POP) {                                       // js is the same in every lane, so these branches are warp-uniform
            if (j0 + G <= js) pre += gsum;
            else if (j0 <= js) {
#pragma unroll
                for (int t = 0; t < G; ++t) {
                    pre += (j0 + t < js) ? vv[t] : 0u;
                    if (j0 + t == js) pv = vv[t];
                }
            }
        }
    };
    if (wide) {
#pragma unroll 1
        for (int j0 = 0; j0 < NB - G; j0 += G) group(j0, std::false_type{}, std::true_type{});
        group(NB - G, std::true_type{}, std::true_type{});
    } else {
#pragma unroll 1
        for (int j0 = 0; j0 < NB - G; j0 += G) group(j0, std::false_type{}, std::false_type{});
        group(NB - G, std::true_type{}, std::false_type{});   // its last bin is the lane's last bin, whose cdf is already known
    }
    int lbi = bestj0;                                     // first position of the maximum inside its group
#pragma unroll
    for (int t = G - 1; t >= 0; --t) if (bestv[t] == lbest) lbi = bestj0 + t;
    uint32_t incl = lsum;
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += t;
    }
    const uint32_t total = __shfl_sync(FULL, incl, 31);
    // :35 first maximum of the row: lanes own ascending blocks, so it is the lowest lane that holds the row maximum
    const uint32_t rowmax = __reduce_max_sync(FULL, lbest);
    const int wl = __ffs(__ballot_sync(FULL, lbest == rowmax)) - 1;
    const int bi = __shfl_sync(FULL, lane * NB + lbi, wl);
    const uint32_t rem = (1u << bits) - total;
    const int64_t out = (int64_t)si * L + row;
    if (POP) {
        constexpr int LPC = 32 / NB;                      // lanes per 32-bin chunk
        const uint32_t base = incl - lsum + ((lane * NB > bi) ? rem : 0u);
        if (lane % LPC == 0) coarse[out * NB + lane / LPC] = base;
        if (lane == 0) fix[out] = make_uint2((uint32_t)bi, rem);
    } else {
        const uint32_t cb = __shfl_sync(FULL, incl - lsum + pre, owner);      // integer cdf at the symbol, before the remnant
        const uint32_t pb = __shfl_sync(FULL, pv, owner);
        if (lane == 0) {
            const uint32_t pf = pb + (bi == sy ? rem : 0u);
            const uint64_t M = pf == 1u ? ~0ull : ~0ull / (uint64_t)pf;      // reciprocal for the serial phase's division
            if ((unsigned)sy >= (unsigned)S) pairs[out] = make_uint4(0u, 0u, 0u, 0u);   // out-of-range symbol: flagged by the serial phase
            else pairs[out] = make_uint4(pf, cb + (bi < sy ? rem : 0u), (uint32_t)M, (uint32_t)(M >> 32));
        }
    }
}

// ---- phase B: push -------------------------------------------------------------------------------------------------
constexpr int BW = 4;
// MASK: rowmask holds L/32 words per stream; bit (i & 31) of word si * L/32 + i/32 clear -> row i of stream si is not
// coded.  (A template flag rather than a NULL test, so that the unmasked kernel is the plain loop: the per-row test cost
// 16 % of this latency-bound kernel when it was always compiled in.)
template <bool MASK>
__global__ void __launch_bounds__(BW * 32) k_push_pairs(bsw_streams sv, int first, int count, const uint4 *__restrict__ pairs,
                                                        int64_t L, int bits, const uint32_t *__restrict__ rowmask) {
    const int lane = threadIdx.x & 31;
    const int si = blockIdx.x * BW + (threadIdx.x >> 5);
    if (si >= count) return;
    const int b = first + si;
    WarpStream2 ws;
    ws.open(sv, b);
    if (ws.err) return;
    ws.push_begin(lane);
    const uint4 *pp = pairs + (int64_t)si * L;
    const uint32_t *rm = MASK ? rowmask + (int64_t)si * (L >> 5) : nullptr;
    uint4 nxt = (lane < L) ? __ldg(pp + lane) : make_uint4(1, 0, 0xffffffffu, 0xffffffffu);
    for (int64_t i0 = 0; i0 < L && !ws.err; i0 += 32) {
        uint4 cur = nxt;
        int64_t r = i0 + 32 + lane;
        if (r < L) nxt = __ldg(pp + r);                   // prefetch the next 32 rows
        const uint32_t live = MASK ? __ldg(rm + (i0 >> 5)) : FULL;
        int n = (int)min((int64_t)32, L - i0);
        for (int j = 0; j < n && !ws.err; ++j) {
            if (MASK && !((live >> j) & 1u)) continue;    // masked row: head and word stack untouched
            uint64_t M = ((uint64_t)__shfl_sync(FULL, cur.w, j) << 32) | __shfl_sync(FULL, cur.z, j);
            const uint32_t pj = __shfl_sync(FULL, cur.x, j);
            if (pj == 0u) { ws.err = BSW_E_INVALID; break; }     // phase A saw a symbol outside the support (reference: IndexError)
            ws.encode_magic(pj, __shfl_sync(FULL, cur.y, j), M, bits, lane);
        }
    }
    ws.push_end(lane);
    ws.close(sv, b, lane);
}

// ---- phase B: pop ----------------------------------------------------------------------------------------------------
template <int NB, bool MASK>
__global__ void __launch_bounds__(BW * 32) k_pop_coarse(bsw_streams sv, int first, int count, const float *__restrict__ mu,
        int64_t mss, const float *__restrict__ sc, int64_t sss, const double *__restrict__ endp, int64_t ers,
        const uint32_t *__restrict__ coarse, const uint2 *__restrict__ fix, int16_t *__restrict__ sym, int64_t L,
        int bits, int q, const uint32_t *__restrict__ rowmask) {
    const int lane = threadIdx.x & 31;
    const int si = blockIdx.x * BW + (threadIdx.x >> 5);
    if (si >= count) return;
    const int b = first + si;
    WarpStream2 ws;
    ws.open(sv, b);
    if (ws.err) return;
    constexpr int S = 32 * NB;
    const float *mub = mu + (int64_t)si * mss, *scb = sc + (int64_t)si * sss;
    const uint32_t *cb = coarse + (int64_t)si * L * NB;
    const uint2 *fb = fix + (int64_t)si * L;
    int16_t *sy = sym + (int64_t)si * L;
    const double mult = (double)(((int64_t)1 << bits) - ((int64_t)1 << q));
    const uint32_t mask = (uint32_t)(((uint64_t)1 << bits) - 1);

    float mu_w = 0.f, sc_w = 1.f;
    uint2 fx_w = make_uint2(0, 0);
    int my_sym = 0;
    // per-row scalars (mu, sigma, argmax, remnant, row mask word) of a block of 32 rows, loaded one block ahead of their use
    float mu_nx, sc_nx;
    uint2 fx_nx;
    const uint32_t *rm = MASK ? rowmask + (int64_t)si * (L >> 5) : nullptr;
    uint32_t live_w = FULL, live_nx;
    {
        int64_t r = ((L - 1) & ~(int64_t)31) + lane;
        mu_nx = r < L ? mub[r] : 0.f;
        sc_nx = r < L ? scb[r] : 1.f;
        fx_nx = r < L ? __ldg(fb + r) : make_uint2(0, 0);
        live_nx = MASK ? __ldg(rm + ((L - 1) >> 5)) : FULL;
    }
    // coarse cdf rows are independent of the head: keep the loads two rows ahead of their use.  (They are issued AFTER
    // the per-row shuffles below: the first version issued the load first and ncu showed every row stalling ~700 cycles
    // on that load's scoreboard at the first shuffle, profiles/r1_ncu_popcoarse.md.)
    uint32_t base_n1 = (lane < NB) ? __ldg(cb + (L - 1) * NB + lane) : 0xffffffffu;
    uint32_t base_n2 = (lane < NB && L > 1) ? __ldg(cb + (L - 2) * NB + lane) : 0xffffffffu;
    for (int64_t i = L - 1; i >= 0; --i) {
        const int j32 = (int)(i & 31);
        const bool new_block = (j32 == 31 || i == L - 1);
        if (new_block) { mu_w = mu_nx; sc_w = sc_nx; fx_w = fx_nx; live_w = live_nx; }
        const double m_ = (double)__shfl_sync(FULL, mu_w, j32), s_ = (double)__shfl_sync(FULL, sc_w, j32);
        const int bi = (int)__shfl_sync(FULL, fx_w.x, j32);
        const uint32_t rem = __shfl_sync(FULL, fx_w.y, j32);
        if (new_block) {                                  // the block below this one
            int64_t r = (i & ~(int64_t)31) - 32 + lane;
            mu_nx = r >= 0 ? mub[r] : 0.f;
            sc_nx = r >= 0 ? scb[r] : 1.f;
            fx_nx = r >= 0 ? __ldg(fb + r) : make_uint2(0, 0);
            if (MASK && i >= 32) live_nx = __ldg(rm + (i >> 5) - 1);
        }
        const uint32_t base = base_n1;
        base_n1 = base_n2;
        if (i > 1) base_n2 = (lane < NB) ? __ldg(cb + (i - 2) * NB + lane) : 0xffffffffu;
        if (MASK && !((live_w >> j32) & 1u)) {            // masked row: nothing decoded, the symbol slot keeps what it held
            if (j32 == 0) {
                const int64_t r = i + lane;
                if (r < L) sy[r] = (int16_t)my_sym;
            }
            continue;
        }
        const double rs = __ddiv_rn(1.0, s_);
        const uint32_t mm = (uint32_t)ws.x & mask;                                       // cifar_compress.py:60
        const int chunk = 31 - __clz(__ballot_sync(FULL, base <= mm));                   // base of lanes >= NB is UINT_MAX
        const int k = chunk * 32 + lane;
        const double *e = endp + i * ers;
        // two independent cdf evaluations per lane (upper and lower endpoint of my bin)
        double c_hi = (k == S - 1) ? 1.0 : bsw_cdf_fast(__ldg(e + k), m_, s_, rs);
        double c_lo = (k == 0) ? 0.0 : bsw_cdf_fast(__ldg(e + k - 1), m_, s_, rs);
        uint32_t v = __double2uint_rz(__dmul_rn(__dsub_rn(c_hi, c_lo), mult)) + 1u + (k == bi ? rem : 0u);
        uint32_t incl = v;
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t t = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += t;
        }
        const uint32_t cex = __shfl_sync(FULL, base, chunk) + incl - v;                  // integer cdf at my bin
        const int js = 31 - __clz(__ballot_sync(FULL, cex <= mm));                       // :61 searchsorted 'right' - 1
        const uint32_t ps = __shfl_sync(FULL, v, js), cs = __shfl_sync(FULL, cex, js);
        if (lane == j32) my_sym = chunk * 32 + js;                                       // :62
        ws.decode(ps, cs, mm, bits, lane);                                               // :63-65
        if (j32 == 0 || ws.err) {
            int64_t r = (i & ~(int64_t)31) + lane;
            if (r < L && r >= i) sy[r] = (int16_t)my_sym;
            if (ws.err) break;
        }
    }
    ws.close(sv, b, lane);
}

// ---- phase B: pop from the full integer table (small batches) --------------------------------------------------------
// Same search as k_pop_coarse, but the 32 integer pmfs of the chosen chunk are read back from phase A's table instead of
// being recomputed: no float64 on the serial path (per row: coarse cdf [prefetched] -> ballot -> one 128-byte load ->
// warp scan -> ballot -> decode).
template <int NB>
__global__ void __launch_bounds__(BW * 32) k_pop_full(bsw_streams sv, int first, int count, const uint32_t *__restrict__ pfull,
        const uint32_t *__restrict__ coarse, const uint2 *__restrict__ fix, int16_t *__restrict__ sym, int64_t L, int bits,
        int shared_tables) {
    const int lane = threadIdx.x & 31;
    const int si = blockIdx.x * BW + (threadIdx.x >> 5);
    if (si >= count) return;
    const int b = first + si;
    WarpStream2 ws;
    ws.open(sv, b);
    if (ws.err) return;
    constexpr int S = 32 * NB;
    const int64_t ts = shared_tables ? 0 : si;            // one table set for every stream (the prior) or one per stream
    const uint32_t *cb = coarse + ts * L * NB;
    const uint32_t *pb = pfull + ts * L * S;
    const uint2 *fb = fix + ts * L;
    int16_t *sy = sym + (int64_t)si * L;
    const uint32_t mask = (uint32_t)(((uint64_t)1 << bits) - 1);
    uint2 fx_w = make_uint2(0, 0), fx_nx;
    int my_sym = 0;
    {
        int64_t r = ((L - 1) & ~(int64_t)31) + lane;
        fx_nx = r < L ? __ldg(fb + r) : make_uint2(0, 0);
    }
    uint32_t base_n1 = (lane < NB) ? __ldg(cb + (L - 1) * NB + lane) : 0xffffffffu;
    uint32_t base_n2 = (lane < NB && L > 1) ? __ldg(cb + (L - 2) * NB + lane) : 0xffffffffu;
    for (int64_t i = L - 1; i >= 0; --i) {
        const int j32 = (int)(i & 31);
        const bool new_block = (j32 == 31 || i == L - 1);
        if (new_block) fx_w = fx_nx;
        const int bi = (int)__shfl_sync(FULL, fx_w.x, j32);
        const uint32_t rem = __shfl_sync(FULL, fx_w.y, j32);
        if (new_block) {
            int64_t r = (i & ~(int64_t)31) - 32 + lane;
            fx_nx = r >= 0 ? __ldg(fb + r) : make_uint2(0, 0);
        }
        const uint32_t base = base_n1;
        base_n1 = base_n2;
        if (i > 1) base_n2 = (lane < NB) ? __ldg(cb + (i - 2) * NB + lane) : 0xffffffffu;
        const uint32_t mm = (uint32_t)ws.x & mask;                                       // cifar_compress.py:60
        const int chunk = 31 - __clz(__ballot_sync(FULL, base <= mm));
        const int k = chunk * 32 + lane;
        uint32_t v = __ldg(pb + i * S + k) + (k == bi ? rem : 0u);
        uint32_t incl = v;
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t t = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += t;
        }
        const uint32_t cex = __shfl_sync(FULL, base, chunk) + incl - v;
        const int js = 31 - __clz(__ballot_sync(FULL, cex <= mm));                       // :61
        const uint32_t ps = __shfl_sync(FULL, v, js), cs = __shfl_sync(FULL, cex, js);
        if (lane == j32) my_sym = chunk * 32 + js;                                       // :62
        ws.decode(ps, cs, mm, bits, lane);                                               // :63-65
        if (j32 == 0 || ws.err) {
            int64_t r = (i & ~(int64_t)31) + lane;
            if (r < L && r >= i) sy[r] = (int16_t)my_sym;
            if (ws.err) break;
        }
    }
    ws.close(sv, b, lane);
}

template <int NB>
int launch_pop_full(bsw_streams *s, int first, int count, const uint32_t *pfull, const uint32_t *coarse, const uint2 *fix,
                    int16_t *sym, int64_t L, int bits, int shared_tables, cudaStream_t st) {
    k_pop_full<NB><<<(count + BW - 1) / BW, BW * 32, 0, st>>>(*s, first, count, pfull, coarse, fix, sym, L, bits, shared_tables);
    BSW_LAUNCH_CHECK();
    return BSW_OK;
}

template <int NB>
int launch_rows(int phase, bool pop, bsw_streams *s, int first, int count, const float *mu, int64_t mss, const float *sc,
                int64_t sss, const double *endp, int64_t ers, int16_t *sym, int64_t L, int bits, int q, void *scratch,
                const uint32_t *rowmask, cudaStream_t st) {
    dim3 grid((unsigned)L, (count + RW - 1) / RW);
    // pop scratch layout: [coarse: count*L*NB u32, rounded up to 8 bytes] [fix: count*L uint2]
    uint4 *pairs = (uint4 *)scratch;
    uint32_t *coarse = (uint32_t *)scratch;
    uint2 *fix = (uint2 *)((uint8_t *)scratch + (((size_t)count * L * NB * 4 + 7) & ~(size_t)7));
    const BswApxRegs kp = bsw_apx_params();
    // BSW_ROWS_EXACT=1: evaluate the exact cdf for every bin instead of screening with bsw_cdf_apx (A/B switch; same output)
    static const bool env_exact = getenv("BSW_ROWS_EXACT") && getenv("BSW_ROWS_EXACT")[0] == '1';
    const bool exact = bits > 31 || env_exact;
    BSW_MAX_SHARED_ONCE((k_rows<NB, true, false>)); BSW_MAX_SHARED_ONCE((k_rows<NB, true, true>));
    BSW_MAX_SHARED_ONCE((k_rows<NB, false, false>)); BSW_MAX_SHARED_ONCE((k_rows<NB, false, true>));
    BSW_MAX_SHARED_ONCE((k_pop_coarse<NB, false>)); BSW_MAX_SHARED_ONCE((k_pop_coarse<NB, true>));
    BSW_MAX_SHARED_ONCE(k_push_pairs<false>); BSW_MAX_SHARED_ONCE(k_push_pairs<true>);
    if (phase == 0) {
        if (pop) {
            if (exact) k_rows<NB, true, false><<<grid, RW * 32, 0, st>>>(count, L, mu, mss, sc, sss, endp, ers, nullptr, bits, q, nullptr, coarse, fix, kp);
            else k_rows<NB, true, true><<<grid, RW * 32, 0, st>>>(count, L, mu, mss, sc, sss, endp, ers, nullptr, bits, q, nullptr, coarse, fix, kp);
        } else {
            if (exact) k_rows<NB, false, false><<<grid, RW * 32, 0, st>>>(count, L, mu, mss, sc, sss, endp, ers, sym, bits, q, pairs, nullptr, nullptr, kp);
            else k_rows<NB, false, true><<<grid, RW * 32, 0, st>>>(count, L, mu, mss, sc, sss, endp, ers, sym, bits, q, pairs, nullptr, nullptr, kp);
        }
    } else {
        const unsigned g = (count + BW - 1) / BW;
        if (pop && rowmask) k_pop_coarse<NB, true><<<g, BW * 32, 0, st>>>(*s, first, count, mu, mss, sc, sss, endp, ers, coarse, fix, sym, L, bits, q, rowmask);
        else if (pop) k_pop_coarse<NB, false><<<g, BW * 32, 0, st>>>(*s, first, count, mu, mss, sc, sss, endp, ers, coarse, fix, sym, L, bits, q, nullptr);
        else if (rowmask) k_push_pairs<true><<<g, BW * 32, 0, st>>>(*s, first, count, pairs, L, bits, rowmask);
        else k_push_pairs<false><<<g, BW * 32, 0, st>>>(*s, first, count, pairs, L, bits, nullptr);
    }
    BSW_LAUNCH_CHECK();
    return BSW_OK;
}

int launch_push_pairs(bsw_streams *s, int first, int count, const void *scratch, int64_t L, int bits, const uint32_t *rowmask,
                      cudaStream_t st) {
    BSW_MAX_SHARED_ONCE(k_push_pairs<false>); BSW_MAX_SHARED_ONCE(k_push_pairs<true>);
    if (rowmask) k_push_pairs<true><<<(count + BW - 1) / BW, BW * 32, 0, st>>>(*s, first, count, (const uint4 *)scratch, L, bits, rowmask);
    else k_push_pairs<false><<<(count + BW - 1) / BW, BW * 32, 0, st>>>(*s, first, count, (const uint4 *)scratch, L, bits, nullptr);
    BSW_LAUNCH_CHECK();
    return BSW_OK;
}

}  // namespace

// Pop from ONE materialised table shared by every stream (the Logistic(0,1) prior): P [L][S] with the remnant already
// applied, coarse[L][S/32] = C[i][32 r], fix = zeros.
__global__ void k_coarse_from_cdf(const uint32_t *__restrict__ C, int64_t L, int S, uint32_t *__restrict__ coarse, uint2 *__restrict__ fix) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int nb = S / 32;
    if (i >= L * nb) return;
    int64_t row = i / nb;
    int r = (int)(i - row * nb);
    coarse[i] = C[row * (S + 1) + 32 * r];
    if (r == 0) fix[row] = make_uint2(0xffffffffu, 0u);
}
int bsw_prior_coarse(const uint32_t *C, int64_t L, int S, uint32_t *coarse, uint2 *fix, cudaStream_t st) {
    int64_t n = L * (S / 32);
    k_coarse_from_cdf<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(C, L, S, coarse, fix);
    BSW_LAUNCH_CHECK();
    return BSW_OK;
}
int bsw_pop_shared_table(bsw_streams *s, int first, int count, const uint32_t *P, const uint32_t *coarse, const uint2 *fix,
                         int16_t *sym, int64_t L, int S, int bits, cudaStream_t st) {
    BSW_REQUIRE(s && first >= 0 && count > 0 && first + count <= s->B, "stream range out of bounds");
    switch (S) {
        case 128:  return launch_pop_full<4>(s, first, count, P, coarse, fix, sym, L, bits, 1, st);
        case 256:  return launch_pop_full<8>(s, first, count, P, coarse, fix, sym, L, bits, 1, st);
        case 512:  return launch_pop_full<16>(s, first, count, P, coarse, fix, sym, L, bits, 1, st);
        case 1024: return launch_pop_full<32>(s, first, count, P, coarse, fix, sym, L, bits, 1, st);
    }
    return BSW_E_INVALID;
}

// ans_rows6.cu
int bsw_rows6_build_meta(const double *endp, int64_t ers, int64_t L, int S, void *meta_dev, int *n_affine_host, cudaStream_t st);
int bsw_rows6_launch(int phase, bool pop, bsw_streams *s, int first, int count, const float *mu, int64_t mss, const float *sc,
                     int64_t sss, const double *endp, int64_t ers, const void *meta, int16_t *sym, int64_t L, int S, int bits,
                     int q, void *scratch, size_t scratch_bytes, const uint32_t *rowmask, cudaStream_t st);

// Scratch bytes of the two-phase coder for `count` streams of L rows: per row 16 B (push: P, C, reciprocal) or
// 136 B (pop: 32 chunk bases + argmax/remnant), whichever kernel family runs.
size_t bsw_rows_scratch_bytes(int count, int64_t L) { return (size_t)count * L * 136; }

// Two-phase variants of bsw_logistic_push / bsw_logistic_pop (same arguments + caller-provided scratch).
// phase 0 = the parallel row-table kernel, phase 1 = the serial coder; call both, in order, on one stream, with the
// same scratch.  meta != NULL selects the affine-row kernels of ans_rows6.cu (meta = bsw_rows6_build_meta of these
// endpoint rows); meta == NULL the generic ones above.
// rowmask (NULL = every row): L/32 words per stream; a clear bit (i & 31) of word i/32 makes the serial phase skip row i --
// the push leaves the state as it is, the pop decodes nothing there and may leave anything in that symbol slot.  Phase A
// still builds the masked rows' tables.
int bsw_logistic_2p(int phase, bool pop, bsw_streams *s, int first, int count, const float *mu, int64_t mss, const float *sc,
                    int64_t sss, const double *endp, int64_t ers, const void *meta, int16_t *sym, int64_t L, int S, int bits,
                    int q, void *scratch, size_t scratch_bytes, const uint32_t *rowmask, cudaStream_t st) {
    BSW_REQUIRE(s && first >= 0 && count > 0 && first + count <= s->B, "stream range out of bounds");
    BSW_REQUIRE(mu && sc && endp && sym && scratch && L > 0 && L < 65536 * 32, "two-phase coder: bad arguments");
    BSW_REQUIRE(ers == 0 || ers >= S, "two-phase coder: endpoint rows must hold S doubles (+1e300 padded)");
    BSW_REQUIRE(scratch_bytes >= (pop ? bsw_rows_scratch_bytes(count, L) : (size_t)count * L * 16), "two-phase coder: scratch too small");
    BSW_REQUIRE((((uintptr_t)scratch) & 15) == 0, "two-phase coder: scratch must be 16-byte aligned");
    BSW_REQUIRE(!rowmask || (L & 31) == 0, "two-phase coder: a row mask needs a multiple of 32 rows");
    if (meta) {
        if (phase == 1 && !pop) return launch_push_pairs(s, first, count, scratch, L, bits, rowmask, st);
        return bsw_rows6_launch(phase, pop, s, first, count, mu, mss, sc, sss, endp, ers, meta, sym, L, S, bits, q, scratch, scratch_bytes, rowmask, st);
    }
    switch (S) {
        case 32:   return launch_rows<1>(phase, pop, s, first, count, mu, mss, sc, sss, endp, ers, sym, L, bits, q, scratch, rowmask, st);
        case 64:   return launch_rows<2>(phase, pop, s, first, count, mu, mss, sc, sss, endp, ers, sym, L, bits, q, scratch, rowmask, st);
        case 128:  return launch_rows<4>(phase, pop, s, first, count, mu, mss, sc, sss, endp, ers, sym, L, bits, q, scratch, rowmask, st);
        case 256:  return launch_rows<8>(phase, pop, s, first, count, mu, mss, sc, sss, endp, ers, sym, L, bits, q, scratch, rowmask, st);
        case 512:  return launch_rows<16>(phase, pop, s, first, count, mu, mss, sc, sss, endp, ers, sym, L, bits, q, scratch, rowmask, st);
        case 1024: return launch_rows<32>(phase, pop, s, first, count, mu, mss, sc, sss, endp, ers, sym, L, bits, q, scratch, rowmask, st);
    }
    bsw_set_error("two-phase coder: support must be one of 32,64,...,1024 (got %d)", S);
    return BSW_E_INVALID;
}

// ---- FP64 peak microbenchmark (roofline denominator of the row-table kernel; MEASURED_PEAKS.json has no FP64 figure) ----
__global__ void k_fp64_peak(double *out, int iters) {
    double a0 = threadIdx.x * 1e-9 + 1.0, a1 = a0 + 1e-3, a2 = a0 + 2e-3, a3 = a0 + 3e-3, a4 = a0 + 4e-3, a5 = a0 + 5e-3,
           a6 = a0 + 6e-3, a7 = a0 + 7e-3;
    const double b = 0.999999999, c = 1e-12;
    for (int i = 0; i < iters; ++i) {
        a0 = fma(a0, b, c); a1 = fma(a1, b, c); a2 = fma(a2, b, c); a3 = fma(a3, b, c);
        a4 = fma(a4, b, c); a5 = fma(a5, b, c); a6 = fma(a6, b, c); a7 = fma(a7, b, c);
    }
    if (a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7 == 12345.678) out[0] = a0;
}
extern "C" int bsw_measure_fp64_peak(double *dfma_per_s) {
    BSW_REQUIRE(dfma_per_s, "null argument");
    double *d = nullptr;
    BSW_CUDA(cudaMalloc(&d, 8));
    int sms = 0;
    BSW_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));
    const int iters = 20000, threads = 512, blocks = sms * 4;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    k_fp64_peak<<<blocks, threads>>>(d, 1000);
    double best = 0;
    for (int rep = 0; rep < 3; ++rep) {
        cudaEventRecord(e0);
        k_fp64_peak<<<blocks, threads>>>(d, iters);
        cudaEventRecord(e1);
        BSW_CUDA(cudaEventSynchronize(e1));
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        double rate = (double)blocks * threads * iters * 8 / (ms * 1e-3);
        if (rate > best) best = rate;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(d);
    *dfma_per_s = best;
    return BSW_OK;
}

// ---- self-test: bsw_cdf_fast against the exact bsw_cdf_div on random (endpoint, mu, sigma) incl. far tails ----
__global__ void k_cdf_selftest(int64_t n, uint64_t seed, unsigned long long *bad, double *worst) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t x = seed + (uint64_t)i * 0x9E3779B97F4A7C15ULL;
    auto nxt = [&]() { x ^= x << 13; x ^= x >> 7; x ^= x << 17; return (double)(x >> 11) * (1.0 / 9007199254740992.0); };
    nxt();
    int mode = (int)(i & 7);
    float scf = (mode < 4) ? (float)(0.1 + 0.9 * nxt()) : (mode < 6 ? (float)(0.00098 + 0.05 * nxt()) : (float)(0.0009 + 2.0 * nxt()));
    float muf = (float)((nxt() - 0.5) * (mode < 4 ? 14.0 : 2.2));
    double e = (nxt() - 0.5) * (mode < 4 ? 14.0 : 2.2);
    if (mode == 7) e = (double)(float)e;
    // (the +inf pad of an endpoint row is never evaluated: kernels use the constant 1 for the last bin)
    double sc = (double)scf, mu = (double)muf, rs = __ddiv_rn(1.0, sc);
    double a = bsw_cdf_fast(e, mu, sc, rs), b = bsw_cdf_div(e, mu, sc);
    double t = __ddiv_rn(__dsub_rn(e, mu), sc);
    bool ok = (a == b) || (fabs(t) >= 690.0 && ((b < 1e-290 && a < 1e-290 && a >= 0.0) || (b == 1.0 && a == 1.0)));
    if (!ok) {
        atomicAdd(bad, 1ULL);
        worst[0] = e; worst[1] = mu; worst[2] = sc; worst[3] = a; worst[4] = b;
    }
}
// ---- self-test of the screening function: worst |bsw_cdf_apx - bsw_cdf_fast| in units of 2^-51 (what the window is in) ----
__global__ void k_cdf_apx_selftest(int64_t n, uint64_t seed, unsigned long long *worst_bits, const BswApxRegs kp) {
    __shared__ double t32[BSW_APX_TABLE_DOUBLES];
    bsw_apx_table_fill(t32, threadIdx.x, blockDim.x);
    __syncthreads();
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t x = seed + (uint64_t)i * 0x9E3779B97F4A7C15ULL;
    auto nxt = [&]() { x ^= x << 13; x ^= x >> 7; x ^= x << 17; return (double)(x >> 11) * (1.0 / 9007199254740992.0); };
    nxt();
    int mode = (int)(i & 7);
    float scf = (mode < 4) ? (float)(0.1 + 0.9 * nxt()) : (mode < 6 ? (float)(0.00098 + 0.05 * nxt()) : (float)(0.0009 + 2.0 * nxt()));
    float muf = (float)((nxt() - 0.5) * (mode < 4 ? 14.0 : 2.2));
    double e = (nxt() - 0.5) * (mode < 4 ? 14.0 : 2.2);
    if (mode == 3) e = muf + (nxt() - 0.5) * 8.0 * scf;                  // the steep part of the curve
    if (mode == 7) e = (double)(float)e;
    double sc = (double)scf, mu = (double)muf, rs = __ddiv_rn(1.0, sc);
    const BswApxRegs KA = kp;
    double a = bsw_cdf_apx<true>(e, mu, rs, smem_u32r(t32) + 8u * (threadIdx.x & 31), KA), b = bsw_cdf_fast(e, mu, sc, rs);
    double err = fabs(a - b) * 2251799813685248.0;                        // 2^51
    if (!(err == err)) err = 1e300;
    atomicMax(worst_bits, (unsigned long long)__double_as_longlong(err));
}
extern "C" int bsw_selftest_cdf_apx(int64_t n, uint64_t seed, double *worst_units_host) {
    BSW_REQUIRE(n > 0 && worst_units_host, "bad arguments");
    unsigned long long *w = nullptr;
    BSW_CUDA(cudaMalloc(&w, 8));
    BSW_CUDA(cudaMemset(w, 0, 8));
    k_cdf_apx_selftest<<<(unsigned)((n + 255) / 256), 256>>>(n, seed, w, bsw_apx_params());
    BSW_LAUNCH_CHECK();
    unsigned long long h = 0;
    BSW_CUDA(cudaMemcpy(&h, w, 8, cudaMemcpyDeviceToHost));
    cudaFree(w);
    memcpy(worst_units_host, &h, 8);
    return BSW_OK;
}
extern "C" int bsw_selftest_cdf(int64_t n, uint64_t seed, int64_t *mismatches_host, double *example_host) {
    BSW_REQUIRE(n > 0 && mismatches_host, "bad arguments");
    unsigned long long *bad = nullptr;
    double *worst = nullptr;
    BSW_CUDA(cudaMalloc(&bad, 8));
    BSW_CUDA(cudaMalloc(&worst, 5 * 8));
    BSW_CUDA(cudaMemset(bad, 0, 8));
    BSW_CUDA(cudaMemset(worst, 0, 40));
    k_cdf_selftest<<<(unsigned)((n + 255) / 256), 256>>>(n, seed, bad, worst);
    BSW_LAUNCH_CHECK();
    unsigned long long h = 0;
    BSW_CUDA(cudaMemcpy(&h, bad, 8, cudaMemcpyDeviceToHost));
    if (example_host) BSW_CUDA(cudaMemcpy(example_host, worst, 40, cudaMemcpyDeviceToHost));
    cudaFree(bad); cudaFree(worst);
    *mismatches_host = (int64_t)h;
    return BSW_OK;
}

// ---- C ABI of the two-phase coder (same contract as bsw_logistic_push/pop + caller-provided scratch) -----------------
// Kernel family for these two entry points: -1 (default) = look at the endpoint rows (one small kernel + a stream
// synchronise) and use the affine-row kernels when every row is a uniform grid, the generic ones otherwise; 0 = generic;
// 1 = affine kernels regardless (rows that are not uniform grids then take their exact path for every bin: correct, slow).
// The codec does not pay the probe: bsw_bins_create classifies every level once.
static int g_rows_mode = -1;
extern "C" int bsw_set_rows_mode(int mode) { g_rows_mode = mode < 0 ? -1 : (mode > 1 ? 1 : mode); return BSW_OK; }
int bsw_rows_mode() {
    static const int env = getenv("BSW_ROWS_MODE") ? atoi(getenv("BSW_ROWS_MODE")) : -1;
    return g_rows_mode >= 0 ? g_rows_mode : (env >= 0 && env <= 1 ? env : -1);
}
extern "C" int64_t bsw_logistic_scratch_bytes(int count, int64_t L, int S, int full_tables) {
    (void)S; (void)full_tables;                           // (the full-table variant of round 1 is gone: same size for every S)
    return (int64_t)(((bsw_rows_scratch_bytes(count, L) + 63) & ~(size_t)63) + (size_t)L * 32 + 64);   // + room for the row metadata
}
static int abi_2p(bool pop, bsw_streams *s, int first, int count, const float *mu, int64_t mss, const float *sc, int64_t sss,
                  const double *endp, int64_t ers, int16_t *sym, int64_t L, int S, int bits, int q, void *scratch,
                  int64_t scratch_bytes, cudaStream_t st) {
    BSW_REQUIRE(scratch && scratch_bytes >= bsw_logistic_scratch_bytes(count, L, S, 0), "two-phase coder: scratch too small");
    const void *meta = nullptr;
    const int mode = bsw_rows_mode();
    if (mode != 0 && S >= 8 && bits >= 8 && bits <= 31) {
        void *m = (uint8_t *)scratch + ((bsw_rows_scratch_bytes(count, L) + 63) & ~(size_t)63);
        int n_aff = 0;
        if (int rc = bsw_rows6_build_meta(endp, ers, L, S, m, mode == 1 ? nullptr : &n_aff, st)) return rc;    // mode 1: no probe, no synchronise
        if (mode == 1 || n_aff == (ers == 0 ? 1 : (int)L)) meta = m;
    }
    const size_t sb = bsw_rows_scratch_bytes(count, L);
    if (int rc = bsw_logistic_2p(0, pop, s, first, count, mu, mss, sc, sss, endp, ers, meta, sym, L, S, bits, q, scratch, sb, nullptr, st)) return rc;
    return bsw_logistic_2p(1, pop, s, first, count, mu, mss, sc, sss, endp, ers, meta, sym, L, S, bits, q, scratch, sb, nullptr, st);
}
extern "C" int bsw_logistic_push_2p(bsw_streams *s, int first, int count, const float *mu, int64_t mss, const float *sc, int64_t sss,
                                    const double *endp, int64_t ers, const int16_t *sym, int64_t L, int S, int bits, int q,
                                    void *scratch, int64_t scratch_bytes, void *stream) {
    return abi_2p(false, s, first, count, mu, mss, sc, sss, endp, ers, (int16_t *)sym, L, S, bits, q, scratch, scratch_bytes, (cudaStream_t)stream);
}
extern "C" int bsw_logistic_pop_2p(bsw_streams *s, int first, int count, const float *mu, int64_t mss, const float *sc, int64_t sss,
                                   const double *endp, int64_t ers, int16_t *sym, int64_t L, int S, int bits, int q,
                                   void *scratch, int64_t scratch_bytes, void *stream) {
    return abi_2p(true, s, first, count, mu, mss, sc, sss, endp, ers, sym, L, S, bits, q, scratch, scratch_bytes, (cudaStream_t)stream);
}
