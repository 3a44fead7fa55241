// Affine-row two-phase logistic coder (sm_100a): the throughput path for every table the reference builds over a UNIFORM
// endpoint grid -- all latent levels below the top one (discretization.py:105-118, KBinsDiscretizer 'uniform') and the
// pixel level (utils/torch/rand.py:146-147).  Same contract and the same integers as k_rows / k_pop_coarse in ans_rows.cu
// (ANS.__init__, cifar_compress.py:25-39; ANS.encode/decode :48-67); what differs is how the float64 work is organised:
//
//   phase A  k_rows6   one warp per stream x eight consecutive rows (four lanes per row).  The plan (rows6_core.cuh) drops
//            the bins whose integer pmf is provably 1 and cuts the live bins [kl,kh) into 32 chunks of m; a lane walks its 8
//            chunks as ONE chain with the geometric recurrence u_{k+4} = u_k rho^4: per bin one multiply, one scaled
//            1 + u (FMA), a Newton reciprocal (3 FMAs) and one add that quantises the scaled cdf -- 6 FP64 instructions --
//            and the pmf is the 64-bit INTEGER difference of two such cdf bit patterns (no shared memory, no endpoint
//            loads).  A bin whose fixed-point pmf lands within `win` of a truncation boundary is recomputed with the
//            exact function bsw_cdf_fast on the real endpoints, so the integers are the exact function's.
//            push: emits (P_s, C_s, M) of the coded symbol (16 B per row).
//            pop : emits the integer cdf at the start of every chunk (32 x 4 B) + (argmax, remnant, kl, kh, m) (8 B).
//   phase B  k_pop6    one warp per stream, serial in the head: ballot over the 32 chunk bases -> the chunk, every lane
//            evaluates ONE bin of it from (t0 + k dt) -- no table, no dependent global load -- scan + ballot -> symbol.
//            (push: k_push_pairs of ans_rows.cu, unchanged.)
//
// HBM traffic per (stream,row): 10 B in (mu, sigma, symbol) + 16 B (push) or 136 B (pop) of scratch written and read once.
#include <stdlib.h>
#include <type_traits>
#include "bsw_common.cuh"
#include "rows6_core.cuh"

#define FULL 0xffffffffu

namespace {

// phase A: 16 warps per CTA (16 streams x the same row group), 64 registers per thread -> two CTAs per SM
constexpr int PW6 = 4;       // warps (= streams) per CTA in phase B

// exact float64 pmf of bin k of the row (what the reference's tensor expression yields, cifar_compress.py:182-184)
__device__ __noinline__ double r6_exact_pmf(const double *__restrict__ e, int k, int S, double m, double s, double rs) {
    const double c = (k == S - 1) ? 1.0 : bsw_cdf_fast(__ldg(e + k), m, s, rs);
    const double p = (k == 0) ? 0.0 : bsw_cdf_fast(__ldg(e + k - 1), m, s, rs);
    return __dsub_rn(c, p);
}
__device__ __forceinline__ uint32_t r6_exact_pm(const double *__restrict__ e, int k, int S, double m, double s, double rs, double mult) {
    return __double2uint_rz(__dmul_rn(r6_exact_pmf(e, k, S, m, s, rs), mult));        // :29 trunc
}
// The rare path of the table kernel: everything it needs is re-derived from its by-value arguments (registers, no stack
// frame in the caller), so that the hot loop does not have to keep mu, sigma, 1/sigma, mult and the endpoint pointer alive.
__device__ __noinline__ double r6_slow_pmf(const float *__restrict__ mu, int64_t mss, const float *__restrict__ sc, int64_t sss,
                                           const double *__restrict__ endp, int64_t ers, int S, int64_t row, int si, int k) {
    const double m = (double)mu[(int64_t)si * mss + row], s = (double)sc[(int64_t)si * sss + row];
    return r6_exact_pmf(endp + row * ers, k, S, m, s, __ddiv_rn(1.0, s));
}

// ---- per-row metadata: least-effort affine fit through the first and last endpoint + its worst deviation ------------------
__global__ void k_row_meta(const double *__restrict__ endp, int64_t ers, int64_t L, int S, R6RowMeta *__restrict__ meta,
                           int *__restrict__ n_affine) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= L) return;
    const double *e = endp + row * ers;
    const int n = S - 1;                                  // real endpoints (entry S-1 of a padded row is the +1e300 pad)
    const double a = e[0], d = (e[n - 1] - a) / (double)(n - 1);
    double dev = 0.0, emax = 0.0;
    for (int k = lane; k < n; k += 32) {
        const double v = e[k];
        dev = fmax(dev, fabs(v - fma((double)k, d, a)));
        emax = fmax(emax, fabs(v));
    }
    for (int o = 16; o; o >>= 1) {
        dev = fmax(dev, __shfl_xor_sync(FULL, dev, o));
        emax = fmax(emax, __shfl_xor_sync(FULL, emax, o));
    }
    dev += emax * 2.3e-16;                                // the fit itself is evaluated with <= 1 ulp of error
    const bool affine = (d > 0.0) && (dev <= 1e-13 * fmax(1.0, emax)) && (emax < 1e6);
    if (lane == 0) {
        R6RowMeta M;
        M.a = a; M.d = d; M.dev = affine ? dev : __longlong_as_double(0x7ff0000000000000LL); M.rsv = 0.0;
        meta[row] = M;
        if (affine) atomicAdd(n_affine, 1);
    }
}

// ---- phase A -------------------------------------------------------------------------------------------------------------
// One warp = one stream x 32/LPR consecutive rows: LPR lanes share a row, and every lane walks CPL = 32/LPR of the row's 32
// chunks (chunks j*CPL .. j*CPL+CPL-1 for lane j of the row: contiguous bins, one chain).  The integers do not depend on
// LPR -- they are the exact function's either way (asserted by the mapping test and the verify build); what LPR buys is
// that the per-row work (1/sigma, the plan, two exps, the scan / argmax / remnant epilogue: about as many instructions as
// 32 bins of the loop) is issued once per 32/LPR rows instead of once per row.  LPR = 32 is one row per warp.
// vstat (VERIFY builds only): [0] bins whose emitted integer differs from the exact function's, [1] worst
// |screened - exact| scaled pmf of a bin that was trusted, in thousandths of that row's window (1000 = the error that
// could flip a truncation), [2] bins checked, [3] bins that took the exact path.
template <bool POP, bool VERIFY, int LPR>
__global__ void __launch_bounds__(512, 2) k_rows6(int count, int64_t L, int S, const float *__restrict__ mu, int64_t mss,
        const float *__restrict__ sc, int64_t sss, const double *__restrict__ endp, int64_t ers,
        const R6RowMeta *__restrict__ meta, int64_t mrs, const int16_t *__restrict__ sym, int bits, int q,
        uint4 *__restrict__ pairs, uint32_t *__restrict__ bases, uint2 *__restrict__ fix, unsigned long long *vstat, int zero,
        double mult2, double rmult2, double Tone) {
    // mult2 = (2^bits - 2^q) * 2^20 (:28; the pmf in 2^-20 fixed point: < 2^51), its reciprocal and Tone = mult2 + 1.5 * 2^52
    // (the quantised cdf of the row's last upper endpoint, cdf = 1: exact) come in as arguments:
    // FP64 instructions read them straight from the constant bank, where a value derived in the kernel was re-derived
    // (2 moves + a DMUL) by the compiler in every 4-bin group to save two registers.
    constexpr int RPW = 32 / LPR;                         // rows per warp
    constexpr int CPL = 32 / LPR;                         // chunks per lane
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int j = lane % LPR;                             // my position among the lanes of my row
    // grid = (groups of RPW rows, groups of 16 streams)
    const int si = blockIdx.y * 16 + warp;
    if (si >= count) return;
    const bool valid = (int64_t)blockIdx.x * RPW + lane / LPR < L;
    const int64_t row = valid ? (int64_t)blockIdx.x * RPW + lane / LPR : L - 1;   // (lanes past the end redo the last row, write nothing)
    R6Plan pl;
    {
        const R6RowMeta M = meta[row * mrs];
        const double m = (double)mu[(int64_t)si * mss + row], s = (double)sc[(int64_t)si * sss + row];   // cifar_train.py:375-376 up-cast
        pl = r6_plan(M, m, __ddiv_rn(1.0, s), S, bits);
    }
    int sy = 0;
    if (!POP) sy = (int)sym[(int64_t)si * L + row];
    auto slow_raw = [&](int k) -> uint32_t {              // the exact function's integer trunc(pmf * mult) (:29)
        const double mult = (double)(((int64_t)1 << bits) - ((int64_t)1 << q));
        return __double2uint_rz(__dmul_rn(r6_slow_pmf(mu, mss, sc, sss, endp, ers, S, row, si, k), mult));
    };

    // The loop works on raw = trunc(pmf * mult); P = raw + 1 (:29, :32) is restored once per lane at the end.
    // My bins: chunks j*CPL .. j*CPL+CPL-1 are contiguous, [ks0, kend), walked as ONE chain of 4-bin groups anchored by a
    // single exp (the 4-step multiplier rho[3] has its own exp, so 64 steps accumulate < 4 of the 64 window units: measured
    // by the CPU model and by the verify build); chunk boundaries only mark where the pop side's chunk bases are taken.
    const int ks0 = pl.kl + j * CPL * pl.m;
    const int kend = min(ks0 + CPL * pl.m, pl.kh);
    uint32_t rsum = 0, lbest = 0, pre = 0, pv = 0, npre = 0;
    bool have_pv = false;
    __shared__ uint4 bestq[512];                          // per thread: the four values of its best group so far (one predicated
    uint32_t bq_addr;                                     // 16-byte store per update instead of four moves); volatile: not re-derived per store
    asm volatile("{\n.reg .u64 t;\ncvta.to.shared.u64 t, %1;\ncvt.u32.u64 %0, t;\n}" : "=r"(bq_addr) : "l"(&bestq[threadIdx.x]));
    int bestk = ks0;
    uint32_t cpre[CPL];                                   // P-sum of my bins before chunk i (for the chunk bases of the pop side)
#pragma unroll
    for (int t = 0; t < CPL; ++t) cpre[t] = 0u;
    if (ks0 < kend) {
        const double rho1 = r6_exp_neg(pl.dt), rho4 = r6_exp_neg(__dmul_rn(4.0, pl.dt));
        // four registers that just hold `zero` (a kernel argument, so the compiler cannot fold it), see r6_rcp_seed_lo
        const int zlo[4] = {zero, zero, zero, zero};
        double ub = r6_exp_neg(__fma_rn((double)(ks0 - 1), pl.dt, pl.t0));       // exp(-t) at the endpoint below my first bin
        double Tprev = ks0 == 0 ? R6_MAGIC0 : r6_quant(ub, rmult2);             // lower edge of bin 0 is cdf = 0 (:184)
        int next_chunk = ks0, ci = 0;
        // one 4-bin group; `last`: the group that ends the row, whose upper edge is cdf = 1 exactly (:184) -- peeled out of the
        // loop below so that the loop does not carry the test and the two selects
        auto group = [&](const int k0, const bool last) __attribute__((always_inline)) {
            if (POP && k0 == next_chunk) {                // chunk boundary: remember the P-sum so far
                const uint32_t sofar = rsum + (uint32_t)(k0 - ks0);
#pragma unroll
                for (int t = 0; t < CPL; ++t) if (t == ci) cpre[t] = sofar;
                ++ci; next_chunk += pl.m;
            }
            uint32_t dlo[4], dhi[4], vv[4];
            r6_group_q(ub, Tprev, rho1, rho4, rmult2, Tone, last, zlo, pl.win, dlo, dhi);
            bool any = false;
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                vv[t] = r6_raw_q(dlo[t], dhi[t]);
                any |= r6_doubt_q(dlo[t], pl.mask);
            }
            // (No test for a negative pmf: on an affine row u decreases strictly along the chain, so T can only fail to
            // increase by rounding noise, one unit -- far inside the window.  Rows the plan does not vouch for have
            // mask == 0 and take the exact path for every bin.)
            if (VERIFY) {
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const double ex = r6_slow_pmf(mu, mss, sc, sss, endp, ers, S, row, si, k0 + t);
                    if (pl.mask != 0u && !r6_doubt_q(dlo[t], pl.mask)) {
                        const double D = (double)(((unsigned long long)dhi[t] << 32) | dlo[t]) - (double)pl.win;
                        const double err = fabs(D - ex * mult2) * 1000.0 / (double)pl.win;
                        atomicMax(vstat + 1, (unsigned long long)(err < 1e18 ? err + 0.999 : 1e18));
                    }
                    atomicAdd(vstat + 2, 1ULL);
                }
            }
            if (any) {
#pragma unroll
                for (int t = 0; t < 4; ++t)
                    if (r6_doubt_q(dlo[t], pl.mask)) {
                        vv[t] = slow_raw(k0 + t);
                        if (VERIFY) atomicAdd(vstat + 3, 1ULL);
                    }
            }
            if (VERIFY) {
#pragma unroll
                for (int t = 0; t < 4; ++t)
                    if (vv[t] != slow_raw(k0 + t)) atomicAdd(vstat, 1ULL);
            }
            const uint32_t gsum = (vv[0] + vv[1]) + (vv[2] + vv[3]);
            const uint32_t gmax = max(max(vv[0], vv[1]), max(vv[2], vv[3]));
            rsum += gsum;
            if (gmax > lbest) {                           // strict: the earlier group keeps a tie (:35 first maximum)
                lbest = gmax; bestk = k0;
                asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(bq_addr), "r"(vv[0]), "r"(vv[1]), "r"(vv[2]), "r"(vv[3]) : "memory");
            }
            if (!POP) {                                   // the group that holds my row's symbol: once per row, in one of its lanes
                if ((unsigned)(sy - k0) < 4u) {
                    pre = rsum - gsum;                    // my bins before this group (rsum already holds the group)
                    npre = (uint32_t)(k0 - ks0);
#pragma unroll
                    for (int t = 0; t < 4; ++t) {
                        if (k0 + t < sy) { pre += vv[t]; ++npre; }
                        if (k0 + t == sy) { pv = vv[t]; have_pv = true; }
                    }
                }
            }
        };
        const int kmain = kend == S ? kend - 4 : kend;
#pragma unroll 2
        for (int k0 = ks0; k0 < kmain; k0 += 4) group(k0, false);
        if (kend == S) group(kend - 4, true);
        if (!POP && sy >= kend) { pre = rsum; npre = (uint32_t)(kend - ks0); }      // all my bins lie below the symbol
        if (POP) {                                        // chunks past my last bin: the P-sum of all my bins
            const uint32_t sofar = rsum + (uint32_t)(kend - ks0);
#pragma unroll
            for (int t = 0; t < CPL; ++t) if (t >= ci) cpre[t] = sofar;
        }
    }
    const uint32_t nbin = ks0 < kend ? (uint32_t)(kend - ks0) : 0u;
    int lbi = bestk;                                      // first position of the maximum inside its group
    if (lbest) {                                          // (no group beat the initial 0: every value is 0, the first bin stands)
        uint4 bq;
        asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(bq.x), "=r"(bq.y), "=r"(bq.z), "=r"(bq.w) : "r"(bq_addr) : "memory");
        const uint32_t bestv[4] = {bq.x, bq.y, bq.z, bq.w};
#pragma unroll
        for (int t = 3; t >= 0; --t) if (bestv[t] == lbest) lbi = bestk + t;
    }
    // back to P = trunc + 1
    const uint32_t lsum = rsum + nbin;
    pre += npre;
    pv += 1u;
    lbest = nbin ? lbest + 1u : 0u;
    uint32_t incl = lsum;
#pragma unroll
    for (int o = 1; o < LPR; o <<= 1) {
        const uint32_t t = __shfl_up_sync(FULL, incl, o, LPR);
        if (j >= o) incl += t;
    }
    // dead bins carry P = 1 each (trunc(...) = 0, +1)
    const uint32_t total = (uint32_t)pl.kl + __shfl_sync(FULL, incl, LPR - 1, LPR) + (uint32_t)(S - pl.kh);
    // :35 first maximum of the row: chunks ascend with the lane, so it is the lowest lane of the row that holds the row maximum
    uint32_t rowmax = lbest;
    int bi = lbi;
#pragma unroll
    for (int o = 1; o < LPR; o <<= 1) {
        const uint32_t ov = __shfl_xor_sync(FULL, rowmax, o, LPR);
        const int ok = __shfl_xor_sync(FULL, bi, o, LPR);
        const bool other_lower = (j & o) != 0;            // my partner is a lower lane: it wins ties
        if (ov > rowmax || (ov == rowmax && other_lower)) { rowmax = ov; bi = ok; }
    }
    const uint32_t rem = (1u << bits) - total;
    const int64_t out = (int64_t)si * L + row;
    const uint32_t excl = (uint32_t)pl.kl + incl - lsum;  // integer cdf at my first bin, before the remnant
    if (POP) {
        uint32_t bs[CPL];
#pragma unroll
        for (int t = 0; t < CPL; ++t) {
            const int ks = pl.kl + (j * CPL + t) * pl.m;
            bs[t] = excl + cpre[t] + ((ks > bi) ? rem : 0u);      // (a chunk past the live range gets the cdf at kh: above any m the search sends there)
        }
        if (valid) {
            uint32_t *bo = bases + out * 32 + j * CPL;
            if constexpr (CPL % 4 == 0) {
#pragma unroll
                for (int t = 0; t < CPL; t += 4) *reinterpret_cast<uint4 *>(bo + t) = make_uint4(bs[t], bs[t + 1], bs[t + 2], bs[t + 3]);
            } else if constexpr (CPL == 2) {
                *reinterpret_cast<uint2 *>(bo) = make_uint2(bs[0], bs[1]);
            } else {
#pragma unroll
                for (int t = 0; t < CPL; ++t) bo[t] = bs[t];
            }
            if (j == 0)
                fix[out] = make_uint2((uint32_t)bi | ((uint32_t)(pl.kl >> 2) << 10) | ((uint32_t)(pl.kh >> 2) << 18) | ((uint32_t)(pl.m >> 2) << 27), rem);
        }
    } else {
        // the row's C_s and P_s: sums over the row's lanes (one lane holds pv; every lane holds its share of the prefix)
        uint32_t cb = pre, pb = have_pv ? pv : 0u;
        uint32_t got = have_pv ? 1u : 0u;
#pragma unroll
        for (int o = 1; o < LPR; o <<= 1) {
            cb += __shfl_xor_sync(FULL, cb, o, LPR);
            pb += __shfl_xor_sync(FULL, pb, o, LPR);
            got += __shfl_xor_sync(FULL, got, o, LPR);
        }
        cb += (uint32_t)pl.kl;
        if (!got) {
            if (sy < pl.kl) { cb = (uint32_t)sy; pb = 1u; }
            else { cb = total - (uint32_t)(S - sy); pb = 1u; }
        }
        if (j == 0 && valid) {
            const uint32_t pf = pb + (bi == sy ? rem : 0u);
            const uint64_t Mg = pf == 1u ? ~0ull : ~0ull / (uint64_t)pf;          // reciprocal for the serial phase's division
            if ((unsigned)sy >= (unsigned)S) pairs[out] = make_uint4(0u, 0u, 0u, 0u);    // out-of-range symbol: flagged by the serial phase
            else pairs[out] = make_uint4(pf, cb + (bi < sy ? rem : 0u), (uint32_t)Mg, (uint32_t)(Mg >> 32));
        }
    }
}

// ---- phase B: pop -----------------------------------------------------------------------------------------------------------
struct WarpStream6 {          // same state handling as ans_kernels.cu's WarpStream (pop side only)
    uint32_t *words;
    uint64_t x;
    int len, wbase, err;
    uint32_t wbuf;
    __device__ __forceinline__ void open(const bsw_streams &sv, int b) {
        words = sv.words + (int64_t)b * sv.cap; x = sv.heads[b]; len = sv.nwords[b];
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
    __device__ __forceinline__ void decode(uint32_t p, uint32_t c, uint32_t m, int bits, int lane) {   // cifar_compress.py:63-65
        x = (uint64_t)p * (x >> bits) + m - c;
        if (x < ((uint64_t)1 << 32)) {
            if (len <= 0) { err = BSW_E_UNDERFLOW; return; }
            x = (x << 32) | pop_word(lane);
        }
    }
};
__device__ __forceinline__ double shfl_d(double v, int src) {
    return __hiloint2double(__shfl_sync(FULL, __double2hiint(v), src), __shfl_sync(FULL, __double2loint(v), src));
}

template <bool MASK>          // MASK: skip the rows whose rowmask bit is clear (a template flag, so the unmasked loop is untouched)
__global__ void __launch_bounds__(PW6 * 32) k_pop6(bsw_streams sv, int first, int count, const float *__restrict__ mu, int64_t mss,
        const float *__restrict__ sc, int64_t sss, const double *__restrict__ endp, int64_t ers,
        const R6RowMeta *__restrict__ meta, int64_t mrs, const uint32_t *__restrict__ bases, const uint2 *__restrict__ fix,
        int16_t *__restrict__ sym, int64_t L, int S, int bits, int q, const uint32_t *__restrict__ rowmask) {
    const int lane = threadIdx.x & 31;
    const int si = blockIdx.x * PW6 + (threadIdx.x >> 5);
    if (si >= count) return;
    const int b = first + si;
    WarpStream6 ws;
    ws.open(sv, b);
    if (ws.err) return;
    const float *mub = mu + (int64_t)si * mss, *scb = sc + (int64_t)si * sss;
    const uint32_t *bb = bases + (int64_t)si * L * 32;
    const uint2 *fb = fix + (int64_t)si * L;
    int16_t *sy = sym + (int64_t)si * L;
    const double mult = (double)(((int64_t)1 << bits) - ((int64_t)1 << q));
    const double mult2 = mult * 1048576.0;
    const uint32_t mask = (uint32_t)(((uint64_t)1 << bits) - 1);

    // per-row scalars of a block of 32 rows (lane j <-> row blk*32 + j), loaded one block ahead of their use; the
    // float64 plan of each row (t0, dt, window) is then computed by its lane, 32 rows in parallel.  The block's row mask
    // word (rowmask: L/32 words per stream, NULL = every row) comes with them: a clear bit skips the row.
    float mu_w = 0.f, sc_w = 1.f, mu_nx, sc_nx;
    uint2 fx_w = make_uint2(0, 0), fx_nx;
    double a_nx, d_nx, dev_nx;
    double t0_w = 0.0, dt_w = 1.0, rs_w = 1.0, magic_w = 0.0;
    uint32_t dmask_w = 0;
    const uint32_t *rm = MASK ? rowmask + (int64_t)si * (L >> 5) : nullptr;
    uint32_t live_w = FULL, live_nx = FULL;
    auto load_block = [&](int64_t r0) {
        const int64_t r = r0 + lane;
        const bool ok = r >= 0 && r < L;
        mu_nx = ok ? mub[r] : 0.f;
        sc_nx = ok ? scb[r] : 1.f;
        fx_nx = ok ? __ldg(fb + r) : make_uint2(0, 0);
        const R6RowMeta *mp = meta + (ok ? r : 0) * mrs;
        a_nx = __ldg(&mp->a); d_nx = __ldg(&mp->d); dev_nx = __ldg(&mp->dev);
        if (MASK && r0 >= 0) live_nx = __ldg(rm + (r0 >> 5));
    };
    auto adopt_block = [&]() {
        mu_w = mu_nx; sc_w = sc_nx; fx_w = fx_nx; live_w = live_nx;
        rs_w = __ddiv_rn(1.0, (double)sc_w);
        R6RowMeta M;
        M.a = a_nx; M.d = d_nx; M.dev = dev_nx; M.rsv = 0.0;
        const R6Plan pl = r6_plan(M, (double)mu_w, rs_w, S, bits);
        t0_w = pl.t0; dt_w = pl.dt; magic_w = pl.magic; dmask_w = pl.mask;
    };
    load_block((L - 1) & ~(int64_t)31);
    int my_sym = 0;
    // chunk bases are independent of the head: keep the loads two rows ahead of their use
    uint32_t base_n1 = __ldg(bb + (L - 1) * 32 + lane);
    uint32_t base_n2 = L > 1 ? __ldg(bb + (L - 2) * 32 + lane) : 0u;
    for (int64_t i = L - 1; i >= 0; --i) {
        const int j32 = (int)(i & 31);
        const bool new_block = (j32 == 31 || i == L - 1);
        if (new_block) { adopt_block(); load_block((i & ~(int64_t)31) - 32); }
        const double t0 = shfl_d(t0_w, j32), dt = shfl_d(dt_w, j32), magic = shfl_d(magic_w, j32);
        const uint32_t dmask = __shfl_sync(FULL, dmask_w, j32);
        const uint32_t fx = __shfl_sync(FULL, fx_w.x, j32), rem = __shfl_sync(FULL, fx_w.y, j32);
        const int bi = (int)(fx & 1023u), kl = (int)((fx >> 10) & 255u) << 2, kh = (int)((fx >> 18) & 511u) << 2, m = (int)((fx >> 27) & 15u) << 2;
        const uint32_t base = base_n1;
        base_n1 = base_n2;
        if (i > 1) base_n2 = __ldg(bb + (i - 2) * 32 + lane);
        if (MASK && !((live_w >> j32) & 1u)) {            // masked row: nothing decoded, the symbol slot keeps what it held
            if (j32 == 0) {
                const int64_t r = i + lane;
                if (r < L) sy[r] = (int16_t)my_sym;
            }
            continue;
        }
        const uint32_t mm = (uint32_t)ws.x & mask;                                       // cifar_compress.py:60
        const uint32_t Ckh = (1u << bits) - (uint32_t)(S - kh);                          // integer cdf at bin kh (dead bins: P = 1)
        uint32_t ps, cs;
        int s;
        if (mm < (uint32_t)kl) { s = (int)mm; ps = 1u; cs = mm; }                        // dead bins on the left: C[k] = k
        else if (mm >= Ckh) { s = kh + (int)(mm - Ckh); ps = 1u; cs = mm; }              // dead bins on the right
        else {
            const int chunk = 31 - __clz(__ballot_sync(FULL, base <= mm));              // empty chunks hold Ckh > mm
            const int k = kl + chunk * m + lane;
            const bool active = lane < m && k < kh;
            const double th = __fma_rn((double)k, dt, t0);                               // t at my bin's upper endpoint
            const double c_hi = (k >= S - 1) ? 1.0 : r6_rcp3(__dadd_rn(1.0, r6_exp_neg(th)));
            const double c_lo = (k <= 0) ? 0.0 : r6_rcp3(__dadd_rn(1.0, r6_exp_neg(__dsub_rn(th, dt))));
            const double z = __fma_rn(__dsub_rn(c_hi, c_lo), mult2, magic);
            uint32_t raw = r6_raw(z);
            const bool doubt = active && (r6_doubt(z, dmask) || raw < 0x80000000u);
            if (__any_sync(FULL, doubt)) {                                               // rare: the exact function on the real endpoints
                const double m_ = (double)__shfl_sync(FULL, mu_w, j32), s_ = (double)__shfl_sync(FULL, sc_w, j32);
                const double rs = shfl_d(rs_w, j32);
                if (doubt) raw = r6_exact_pm(endp + i * ers, k, S, m_, s_, rs, mult) + 0x80000000u;
            }
            const uint32_t v = active ? (raw + 0x80000001u) + (k == bi ? rem : 0u) : 0u;  // :29 trunc, :32 +1, :35 remnant
            uint32_t incl = v;
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(FULL, incl, o);
                if (lane >= o) incl += t;
            }
            const uint32_t cex = __shfl_sync(FULL, base, chunk) + incl - v;              // integer cdf at my bin
            const int js = 31 - __clz(__ballot_sync(FULL, active && cex <= mm));         // :61 searchsorted 'right' - 1
            ps = __shfl_sync(FULL, v, js); cs = __shfl_sync(FULL, cex, js);
            s = kl + chunk * m + js;
        }
        if (lane == j32) my_sym = s;                                                     // :62
        ws.decode(ps, cs, mm, bits, lane);                                               // :63-65
        if (j32 == 0 || ws.err) {
            const int64_t r = (i & ~(int64_t)31) + lane;
            if (r < L && r >= i) sy[r] = (int16_t)my_sym;
            if (ws.err) break;
        }
    }
    ws.close(sv, b, lane);
}

unsigned long long *g_vstat = nullptr;                   // device [4], allocated on first use of the VERIFY build
int g_verify = 0;
int g_lpr = 0;                                           // lanes per row of k_rows6 (0: BSW_R6_LPR or the default 4)

}  // namespace

// ---- host side ---------------------------------------------------------------------------------------------------------------
// meta_dev: L entries (or 1 when endp row stride is 0).  n_affine_host (may be NULL) receives the number of rows the
// fast path applies to; the call synchronises `st` only when it is given.
int bsw_rows6_build_meta(const double *endp, int64_t ers, int64_t L, int S, void *meta_dev, int *n_affine_host, cudaStream_t st) {
    BSW_REQUIRE(endp && meta_dev && L > 0 && S >= 8, "bsw_rows6_build_meta: bad arguments");
    const int64_t rows = ers == 0 ? 1 : L;
    static int *cnt = nullptr;                            // (one counter per process: only read back when the caller asks)
    if (!cnt) BSW_CUDA(cudaMalloc(&cnt, sizeof(int)));
    BSW_CUDA(cudaMemsetAsync(cnt, 0, sizeof(int), st));
    k_row_meta<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(endp, ers, rows, S, (R6RowMeta *)meta_dev, cnt);
    BSW_LAUNCH_CHECK();
    if (n_affine_host) {
        int h = 0;
        BSW_CUDA(cudaMemcpyAsync(&h, cnt, sizeof(int), cudaMemcpyDeviceToHost, st));
        BSW_CUDA(cudaStreamSynchronize(st));
        *n_affine_host = h;
    }
    return BSW_OK;
}

size_t bsw_rows6_scratch_bytes(int count, int64_t L) {
    return (size_t)count * L * (32 * 4 + 8);              // pop: 32 chunk bases + fix; push needs 16 B per row
}

int bsw_rows6_launch(int phase, bool pop, bsw_streams *s, int first, int count, const float *mu, int64_t mss, const float *sc,
                     int64_t sss, const double *endp, int64_t ers, const void *meta, int16_t *sym, int64_t L, int S, int bits,
                     int q, void *scratch, size_t scratch_bytes, const uint32_t *rowmask, cudaStream_t st) {
    BSW_REQUIRE(S >= 8 && S <= 1024 && (S & 3) == 0, "affine coder: support must be a multiple of 4 in [8, 1024]");
    BSW_REQUIRE(bits >= 8 && bits <= 31 && q >= 0 && q < bits, "affine coder: bits/quantbits out of range");
    BSW_REQUIRE(scratch_bytes >= (pop ? bsw_rows6_scratch_bytes(count, L) : (size_t)count * L * 16), "affine coder: scratch too small");
    const R6RowMeta *mt = (const R6RowMeta *)meta;
    const int64_t mrs = ers == 0 ? 0 : 1;
    uint4 *pairs = (uint4 *)scratch;
    uint32_t *bases = (uint32_t *)scratch;
    uint2 *fix = (uint2 *)((uint8_t *)scratch + (size_t)count * L * 128);
    if (phase == 0) {
        // BSW_R6_LPR = lanes per row (32, 8, 4 or 2; default 4 = eight rows per warp): same integers, different mapping (A/B runs)
        static const int env_lpr0 = getenv("BSW_R6_LPR") ? atoi(getenv("BSW_R6_LPR")) : 4;
        const int env_lpr = g_lpr > 0 ? g_lpr : env_lpr0;
        if (g_verify && !g_vstat) { BSW_CUDA(cudaMalloc(&g_vstat, 32)); BSW_CUDA(cudaMemset(g_vstat, 0, 32)); }
#define R6_LAUNCH(POP_, VER_, LPR_)                                                                                             \
    BSW_MAX_SHARED_ONCE((k_rows6<POP_, VER_, LPR_>));                                                                             \
    k_rows6<POP_, VER_, LPR_><<<dim3((unsigned)((L + 32 / LPR_ - 1) / (32 / LPR_)), (count + 15) / 16), 512, 0, st>>>(            \
        count, L, S, mu, mss, sc, sss, endp, ers, mt, mrs, POP_ ? nullptr : sym, bits, q, POP_ ? nullptr : pairs,                 \
        POP_ ? bases : nullptr, POP_ ? fix : nullptr, VER_ ? g_vstat : nullptr, 0,                                                \
        (double)(((int64_t)1 << bits) - ((int64_t)1 << q)) * 1048576.0,                                                           \
        1.0 / ((double)(((int64_t)1 << bits) - ((int64_t)1 << q)) * 1048576.0),                                                     \
        (double)(((int64_t)1 << bits) - ((int64_t)1 << q)) * 1048576.0 + R6_MAGIC0)
#define R6_PICK(VER_, LPR_) do { if (pop) { R6_LAUNCH(true, VER_, LPR_); } else { R6_LAUNCH(false, VER_, LPR_); } } while (0)
        if (g_verify) { if (env_lpr == 32) R6_PICK(true, 32); else R6_PICK(true, 4); }
        else if (env_lpr == 32) R6_PICK(false, 32);
        else if (env_lpr == 8) R6_PICK(false, 8);
        else if (env_lpr == 2) R6_PICK(false, 2);
        else R6_PICK(false, 4);
#undef R6_PICK
#undef R6_LAUNCH
    } else {
        BSW_REQUIRE(pop, "affine coder: phase B of a push is k_push_pairs");
        BSW_MAX_SHARED_ONCE(k_pop6<false>); BSW_MAX_SHARED_ONCE(k_pop6<true>);
        if (rowmask) k_pop6<true><<<(count + PW6 - 1) / PW6, PW6 * 32, 0, st>>>(*s, first, count, mu, mss, sc, sss, endp, ers, mt, mrs, bases, fix, sym, L, S, bits, q, rowmask);
        else k_pop6<false><<<(count + PW6 - 1) / PW6, PW6 * 32, 0, st>>>(*s, first, count, mu, mss, sc, sss, endp, ers, mt, mrs, bases, fix, sym, L, S, bits, q, nullptr);
    }
    BSW_LAUNCH_CHECK();
    return BSW_OK;
}

// Debug switch: 1 = every k_rows6 launch also evaluates the exact function for every bin and counts disagreements
// (slow; tests/test_ans_gpu.py runs a full-size level through it).  Read + reset the counters with bsw_rows6_verify_read.
extern "C" int bsw_rows6_set_lanes_per_row(int lpr) {
    BSW_REQUIRE(lpr == 0 || lpr == 2 || lpr == 4 || lpr == 8 || lpr == 32, "bsw_rows6_set_lanes_per_row: 0 (default), 2, 4, 8 or 32");
    g_lpr = lpr;
    return BSW_OK;
}
extern "C" int bsw_rows6_set_verify(int on) { g_verify = on ? 1 : 0; return BSW_OK; }
extern "C" int bsw_rows6_verify_read(uint64_t *out4_host) {
    BSW_REQUIRE(out4_host, "null argument");
    for (int i = 0; i < 4; ++i) out4_host[i] = 0;
    if (!g_vstat) return BSW_OK;
    BSW_CUDA(cudaDeviceSynchronize());
    BSW_CUDA(cudaMemcpy(out4_host, g_vstat, 32, cudaMemcpyDeviceToHost));
    BSW_CUDA(cudaMemset(g_vstat, 0, 32));
    return BSW_OK;
}
