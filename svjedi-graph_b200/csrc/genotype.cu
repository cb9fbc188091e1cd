// Kernel 4: genotype likelihoods, GT and PL per SV from the REF/ALT hit counters.
//
// Restates predict-genotype.py:281-346 (likelihood, allele_normalization,
// encode_genotype) and the gate at :216.  The reference sums binary64 products
// as 28-digit Decimals and truncates -10*(lik+comb) to an int.  Here every
// product is formed with one IEEE multiply (the same double the reference
// holds), converted EXACTLY to 192-bit fixed point (LSB 2^-112) and summed,
// multiplied by 10 and truncated in integer arithmetic — no rounding anywhere,
// which is what the Decimal path amounts to (DESIGN.md, "PL exactness").
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>
#include <string>

#include "svjg_internal.h"

namespace {

constexpr int FRAC_BITS = 112;

struct F192 {   // two's complement, little-endian limbs
    uint64_t w0, w1, w2;
};

__device__ __forceinline__ F192 f_add(const F192 &x, const F192 &y) {
    F192 r;
    r.w0 = x.w0 + y.w0;
    uint64_t c0 = r.w0 < x.w0;
    r.w1 = x.w1 + y.w1;
    uint64_t c1 = r.w1 < x.w1;
    r.w1 += c0;
    c1 |= (r.w1 < c0);
    r.w2 = x.w2 + y.w2 + c1;
    return r;
}
__device__ __forceinline__ F192 f_neg(const F192 &x) {
    F192 n{~x.w0, ~x.w1, ~x.w2};
    return f_add(n, F192{1, 0, 0});
}
__device__ __forceinline__ F192 f_shl(const F192 &x, int s) {   // 0 < s < 64
    return F192{x.w0 << s, (x.w1 << s) | (x.w0 >> (64 - s)), (x.w2 << s) | (x.w1 >> (64 - s))};
}
__device__ __forceinline__ int f_cmp(const F192 &x, const F192 &y) {   // signed
    int64_t xs = int64_t(x.w2), ys = int64_t(y.w2);
    if (xs != ys) return xs < ys ? -1 : 1;
    if (x.w1 != y.w1) return x.w1 < y.w1 ? -1 : 1;
    if (x.w0 != y.w0) return x.w0 < y.w0 ? -1 : 1;
    return 0;
}

// exact conversion; ok=false if the value does not fit the format (never for
// the magnitudes this path produces, see DESIGN.md)
__device__ F192 f_from_double(double d, bool &ok) {
    uint64_t bits = (uint64_t)__double_as_longlong(d);
    uint64_t frac = bits & 0xFFFFFFFFFFFFFull;
    int ex = int((bits >> 52) & 0x7FF);
    bool neg = bits >> 63;
    if (ex == 0x7FF) {
        ok = false;
        return F192{0, 0, 0};
    }
    uint64_t m = ex ? (frac | (1ull << 52)) : frac;
    int q = (ex ? ex : 1) - 1075;            // value = m * 2^q
    if (m == 0) return F192{0, 0, 0};
    int sh = q + FRAC_BITS;
    F192 r{0, 0, 0};
    if (sh < 0) {
        if (sh <= -64 || (m & ((1ull << -sh) - 1))) ok = false;
        r.w0 = sh <= -64 ? 0 : m >> -sh;
    } else if (sh > 190 - 53) {
        ok = false;
    } else {
        int limb = sh >> 6, s = sh & 63;
        uint64_t lo = m << s, hi = s ? m >> (64 - s) : 0;
        if (limb == 0) {
            r.w0 = lo;
            r.w1 = hi;
        } else if (limb == 1) {
            r.w1 = lo;
            r.w2 = hi;
        } else {
            r.w2 = lo;
        }
    }
    return neg ? f_neg(r) : r;
}

// int(-10 * x) with truncation toward zero
__device__ int64_t pl_of(const F192 &x) {
    F192 v = f_add(f_shl(x, 3), f_shl(x, 1));          // 10 x
    bool neg = int64_t(v.w2) < 0;
    F192 mag = neg ? f_neg(v) : v;
    // mag >> 112
    uint64_t q = (mag.w1 >> 48) | (mag.w2 << 16);
    return neg ? int64_t(q) : -int64_t(q);
}

// The genotype of one SV of one sample from its two counters: the gate of predict-genotype.py:216,
// allele_normalization, the likelihoods, the unique argmax, -ms, the rounded counts, log10 C(n, k) and PL.
// Results go to gt[o], flags[o], ad2[2o..], pl[3o..]; k_override[o] is read when k_override is given.
// PLOIDY: the cell has `ploidy` copies (else 2, and `ploidy` is not read: the plain instance is the reference's diploid
// call statement for statement).  Ploidy 1 calls between the "REF" and "ALT" sums L0 and L2 only (gt SVJG_GT_HAP_REF /
// _HAP_ALT / _HAP_MISSING); ploidy 0 makes no call and computes no likelihood, but keeps DP and AD (SVJG_GT_NO_CALL).
// DESIGN.md §8a, "Sex-chromosome ploidy".
template <bool PLOIDY>
__device__ __forceinline__ void genotype_one(uint32_t n0, uint32_t n1, uint32_t idx, uint32_t ty, int64_t min_support,
                                             double la, double lb, double lh, const double *lut, uint32_t lut_nmax,
                                             const double *k_override, size_t o, int64_t *pl, uint8_t *gt,
                                             uint32_t *ad2, uint8_t *flags, uint32_t ploidy) {
    // predict-genotype.py:216 — a key is "in the dict" once it has at least one hit
    bool gate = (ty & 0x3F) <= 3 && !(ty & 0x80) && ty != 255 && idx != 0xFFFFFFFFu && ((n0 | n1) != 0 || (ty & 0x40));
    if (!gate) {
        if constexpr (PLOIDY) gt[o] = ploidy == 2 ? 3 : ploidy == 1 ? SVJG_GT_HAP_MISSING : SVJG_GT_NO_CALL;
        else gt[o] = 3;
        flags[o] = 0;
        ad2[2 * o] = 0;
        ad2[2 * o + 1] = 0;
        pl[3 * o] = pl[3 * o + 1] = pl[3 * o + 2] = 0;
        return;
    }
    ty &= 0x3F;
    // allele_normalization (:327-338): counts in half units
    uint64_t t1 = 2ull * n0, t2 = 2ull * n1;
    uint32_t fl = SVJG_GT_GENOTYPED;
    if (ty == 0 && n0 > 0) {
        t1 = n0;
        fl |= SVJG_GT_HALVED_0;
    } else if (ty == 1 && n1 > 0) {
        t2 = n1;
        fl |= SVJG_GT_HALVED_1;
    }
    if constexpr (PLOIDY) {
        if (ploidy == 0) {
            gt[o] = SVJG_GT_NO_CALL;
            flags[o] = uint8_t(fl);
            ad2[2 * o] = uint32_t(t1);
            ad2[2 * o + 1] = uint32_t(t2);
            pl[3 * o] = pl[3 * o + 1] = pl[3 * o + 2] = 0;
            return;
        }
    }
    double c1 = double(t1) * 0.5, c2 = double(t2) * 0.5, cs = double(t1 + t2) * 0.5;   // exact
    bool ok = true;
    // :295-297 — each product is the double the reference computes
    F192 l0 = f_add(f_from_double(__dmul_rn(c1, la), ok), f_from_double(__dmul_rn(c2, lb), ok));
    F192 l1 = f_from_double(__dmul_rn(cs, lh), ok);
    F192 l2 = f_add(f_from_double(__dmul_rn(c2, la), ok), f_from_double(__dmul_rn(c1, lb), ok));
    // unique argmax (:301-307)
    int c01 = f_cmp(l0, l1), c02 = f_cmp(l0, l2), c12 = f_cmp(l1, l2);
    uint32_t g = 3;
    if (c01 > 0 && c02 > 0) g = 0;
    else if (c01 < 0 && c12 > 0) g = 1;
    else if (c02 < 0 && c12 < 0) g = 2;
    if (int64_t(t1 + t2) < 2 * min_support) g = 3;                                       // :310
    if constexpr (PLOIDY) {
        if (ploidy == 1) {   // the same rule restricted to {L0, L2}
            g = c02 > 0 ? SVJG_GT_HAP_REF : c02 < 0 ? SVJG_GT_HAP_ALT : SVJG_GT_HAP_MISSING;
            if (int64_t(t1 + t2) < 2 * min_support) g = SVJG_GT_HAP_MISSING;
        }
    }
    // rc = int(round(c, 0)), half to even (:291-292)
    uint64_t r1 = (t1 >> 1) + ((t1 & 1) ? ((t1 >> 1) & 1) : 0);
    uint64_t r2 = (t2 >> 1) + ((t2 & 1) ? ((t2 >> 1) & 1) : 0);
    uint64_t nn = r1 + r2;
    double kval;
    bool have_k = false;
    if (k_override) {
        double ko = k_override[o];
        if (ko == ko) {
            kval = ko;
            have_k = true;
        }
    }
    if (!have_k && nn <= lut_nmax) {
        kval = lut[nn * (nn + 1) / 2 + r1];
        have_k = true;
    }
    int64_t p0 = 0, p1 = 0, p2 = 0;
    if (have_k) {
        F192 k = f_from_double(kval, ok);                                                // :313
        p0 = pl_of(f_add(l0, k));
        p1 = pl_of(f_add(l1, k));
        p2 = pl_of(f_add(l2, k));
    } else {
        fl |= SVJG_GT_NEED_K;
    }
    if (!ok) fl |= SVJG_GT_NEED_K;   // out-of-format value: never produce a wrong PL silently
    gt[o] = uint8_t(g);
    flags[o] = uint8_t(fl);
    ad2[2 * o] = uint32_t(t1);
    ad2[2 * o + 1] = uint32_t(t2);
    pl[3 * o] = p0;
    pl[3 * o + 1] = p1;
    pl[3 * o + 2] = p2;
}

// Counters of all ranks, read where they lie: every rank's exchange region is mapped into this
// process (CUDA IPC, NVLink peer access).  The kernel first waits until every rank has signalled
// that its filter is done for this step, then every thread sums the per-rank counters of its SV --
// the all-reduce and the genotype step are one kernel, and only the counters that are needed cross
// the links.
constexpr int XCHG_MAX = 16;
constexpr uint32_t XCHG_FLAG_WORDS = 64;           // arrive[rank] ... arrive[63] = time-out marker
struct Xchg {
    const uint32_t *counts[XCHG_MAX];              // this step's counter buffer of every rank
    volatile uint32_t *flags[XCHG_MAX];            // flag words of every rank's region ([rank] = own)
    uint32_t world, rank, epoch;
    uint32_t signal;                               // 1: this kernel also announces this rank's counters (svjg_xchg_signal not called)
};

template <bool XCHG>
__global__ void genotype_kernel(const uint32_t *__restrict__ counts, const __grid_constant__ Xchg xc,
                                const uint32_t *__restrict__ sv_index,
                                const uint8_t *__restrict__ svtype, uint32_t n, int64_t min_support, double la,
                                double lb, double lh, const double *__restrict__ lut, uint32_t lut_nmax,
                                const double *__restrict__ k_override, int64_t *__restrict__ pl,
                                uint8_t *__restrict__ gt, uint32_t *__restrict__ ad2, uint8_t *__restrict__ flags) {
    if (XCHG) {
        if (threadIdx.x < xc.world) {
            // the counters of this rank were written by kernels in front of this one on the stream:
            // block 0 tells every rank so, then every block waits for the word of every rank
            if (xc.signal && blockIdx.x == 0) {
                __threadfence_system();
                xc.flags[threadIdx.x][xc.rank] = xc.epoch;
            }
            volatile uint32_t *mine = xc.flags[xc.rank];
            const long long t0 = clock64();
            while (mine[threadIdx.x] < xc.epoch) {
                if (clock64() - t0 > 4000000000ll) {                      // ~2 s: a rank is gone; say so, do not hang
                    mine[XCHG_FLAG_WORDS - 1] = 0xDEADu;
                    break;
                }
            }
            __threadfence_system();
        }
        __syncthreads();
    }
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t idx = sv_index[i];
    uint32_t ty = svtype[i];
    uint32_t n0 = 0, n1 = 0;
    if (idx != 0xFFFFFFFFu) {
        if (XCHG) {
            for (uint32_t q = 0; q < xc.world; ++q) {
                const uint2 c = __ldcg(reinterpret_cast<const uint2 *>(xc.counts[q] + 2 * size_t(idx)));
                n0 += c.x;
                n1 += c.y;
            }
        } else {
            uint2 c = *reinterpret_cast<const uint2 *>(counts + 2 * size_t(idx));
            n0 = c.x;
            n1 = c.y;
        }
    }
    genotype_one<false>(n0, n1, idx, ty, min_support, la, lb, lh, lut, lut_nmax, k_override, i, pl, gt, ad2, flags, 2);
}

// One thread per cell (record i, sample s) of a block of records.  The counters are the cohort's sample-major
// matrix ([S][num_sv][2], as the filter writes a sample's counters); the results are record-major ([n][S], the
// order of the VCF text).  PLOIDY: the cell's ploidy is ptab[rclass[i]][sex[s]] (ptab [classes][n_sexes]); without
// it every cell is diploid and the three arrays are not read.
template <bool PLOIDY>
__global__ void genotype_cohort_kernel(const uint32_t *__restrict__ counts, uint32_t num_sv, uint32_t n_samples,
                                       const uint32_t *__restrict__ sv_index, const uint8_t *__restrict__ svtype,
                                       uint32_t n_cells, int64_t min_support, double la, double lb, double lh,
                                       const double *__restrict__ lut, uint32_t lut_nmax, int64_t *__restrict__ pl,
                                       uint8_t *__restrict__ gt, uint32_t *__restrict__ ad2, uint8_t *__restrict__ flags,
                                       const uint8_t *__restrict__ rclass, const uint8_t *__restrict__ sex,
                                       const uint8_t *__restrict__ ptab, uint32_t n_sexes) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_cells) return;
    const uint32_t i = c / n_samples, s = c - i * n_samples;
    const uint32_t idx = sv_index[i];
    uint32_t n0 = 0, n1 = 0;
    if (idx != 0xFFFFFFFFu) {
        const uint2 v = *reinterpret_cast<const uint2 *>(counts + (size_t(s) * num_sv + idx) * 2);
        n0 = v.x;
        n1 = v.y;
    }
    const uint32_t ploidy = PLOIDY ? uint32_t(ptab[rclass[i] * n_sexes + sex[s]]) : 2u;
    genotype_one<PLOIDY>(n0, n1, idx, svtype[i], min_support, la, lb, lh, lut, lut_nmax, nullptr, c, pl, gt, ad2, flags,
                         ploidy);
}

// One term step of the Wigginton-Cutler-Abecasis walk: v * D / E with D and E exact integers (below 2^53), each
// operation one IEEE double rounded to nearest (the Python statement computes the same doubles, DESIGN.md §8a).
__device__ __forceinline__ double hwe_step(double v, uint64_t d, uint64_t e) {
    return __ddiv_rn(__dmul_rn(v, double(d)), double(e));
}

// HWE exact test and excess-heterozygosity p of r0 / h / r2 genotype counts (Wigginton, Cutler & Abecasis 2005) in
// the streaming form of DESIGN.md §8a: the terms, indexed by het count k, are walked down from `mid`, then up from
// it, twice.  Pass 1 sums them all (and those with k >= h); pass 2 sums those no larger than the observed one.  A
// walk stops at its first zero term: every later one is zero too, and adding zero changes no sum.
__device__ void site_exact_tests(uint32_t r0, uint32_t h, uint32_t r2, double &hwe, double &exchet) {
    const uint64_t N = uint64_t(r0) + h + r2;
    const uint64_t rare = 2ull * min(r0, r2) + h;
    if (rare == 0) {                                   // N == 0 included
        hwe = exchet = 1.0;
        return;
    }
    uint64_t mid = rare * (2 * N - rare) / (2 * N);
    if ((mid ^ rare) & 1) ++mid;
    double sum = 1.0, acc_exc = mid >= h ? 1.0 : 0.0, v_obs = mid == h ? 1.0 : 0.0;
    for (int pass = 0; pass < 2; ++pass) {
        double acc_hwe = 1.0 <= v_obs ? 1.0 : 0.0;
        {   // down
            uint64_t k = mid, homr = (rare - mid) / 2, homc = N - mid - homr;
            double v = 1.0;
            while (k >= 2) {
                v = hwe_step(v, k * (k - 1), 4 * (homr + 1) * (homc + 1));
                k -= 2;
                ++homr;
                ++homc;
                if (pass == 0) {
                    sum = __dadd_rn(sum, v);
                    if (k >= h) acc_exc = __dadd_rn(acc_exc, v);
                    if (k == h) v_obs = v;
                } else if (v <= v_obs) {
                    acc_hwe = __dadd_rn(acc_hwe, v);
                }
                if (v == 0.0) break;
            }
        }
        {   // up
            uint64_t k = mid, homr = (rare - mid) / 2, homc = N - mid - homr;
            double v = 1.0;
            while (k + 2 <= rare) {
                v = hwe_step(v, 4 * homr * homc, (k + 2) * (k + 1));
                k += 2;
                --homr;
                --homc;
                if (pass == 0) {
                    sum = __dadd_rn(sum, v);
                    if (k >= h) acc_exc = __dadd_rn(acc_exc, v);
                    if (k == h) v_obs = v;
                } else if (v <= v_obs) {
                    acc_hwe = __dadd_rn(acc_hwe, v);
                }
                if (v == 0.0) break;
            }
        }
        if (pass == 1) hwe = fmin(1.0, __ddiv_rn(acc_hwe, sum));
    }
    exchet = fmin(1.0, __ddiv_rn(acc_exc, sum));
}

// Site statistics of a block of records from the genotype codes the cohort kernel left on the device ([n][S]).
// A block of SITE_THREADS records: each warp counts the 0/0, 0/1 and 1/1 cells of its records (coalesced byte loads
// along the row, one warp reduction per code), then every thread runs the exact tests of one record, which are serial
// per record.  Results: gcount[i] = (r0, h, r2, missing), or with PLOIDY (r0, h, r2, a0, a1, missing) where a0 / a1
// count the haploid calls; hwe[i], exchet[i] of (r0, h, r2).
constexpr int SITE_THREADS = 256;
template <bool PLOIDY>
__global__ void __launch_bounds__(SITE_THREADS)
cohort_site_stats_kernel(const uint8_t *__restrict__ gt, uint32_t n, uint32_t n_samples, uint32_t *__restrict__ gcount,
                         double *__restrict__ hwe, double *__restrict__ exchet) {
    __shared__ uint32_t cnt[PLOIDY ? 5 : 3][SITE_THREADS];
    const uint32_t base = blockIdx.x * SITE_THREADS, lane = threadIdx.x & 31;
    for (uint32_t r = threadIdx.x >> 5; r < SITE_THREADS && base + r < n; r += SITE_THREADS / 32) {
        const uint8_t *row = gt + size_t(base + r) * n_samples;
        uint32_t c0 = 0, c1 = 0, c2 = 0, a0 = 0, a1 = 0;
        for (uint32_t s = lane; s < n_samples; s += 32) {
            const uint32_t g = row[s];
            c0 += g == 0;
            c1 += g == 1;
            c2 += g == 2;
            if constexpr (PLOIDY) {
                a0 += g == SVJG_GT_HAP_REF;
                a1 += g == SVJG_GT_HAP_ALT;
            }
        }
        c0 = __reduce_add_sync(0xFFFFFFFFu, c0);
        c1 = __reduce_add_sync(0xFFFFFFFFu, c1);
        c2 = __reduce_add_sync(0xFFFFFFFFu, c2);
        if constexpr (PLOIDY) {
            a0 = __reduce_add_sync(0xFFFFFFFFu, a0);
            a1 = __reduce_add_sync(0xFFFFFFFFu, a1);
        }
        if (lane == 0) {
            cnt[0][r] = c0;
            cnt[1][r] = c1;
            cnt[2][r] = c2;
            if constexpr (PLOIDY) {
                cnt[3][r] = a0;
                cnt[4][r] = a1;
            }
        }
    }
    __syncthreads();
    const uint32_t i = base + threadIdx.x;
    if (i >= n) return;
    const uint32_t r0 = cnt[0][threadIdx.x], h = cnt[1][threadIdx.x], r2 = cnt[2][threadIdx.x];
    if constexpr (PLOIDY) {
        const uint32_t a0 = cnt[3][threadIdx.x], a1 = cnt[4][threadIdx.x];
        uint2 *g = reinterpret_cast<uint2 *>(gcount + 6 * size_t(i));
        g[0] = make_uint2(r0, h);
        g[1] = make_uint2(r2, a0);
        g[2] = make_uint2(a1, n_samples - r0 - h - r2 - a0 - a1);
    } else {
        reinterpret_cast<uint4 *>(gcount)[i] = make_uint4(r0, h, r2, n_samples - r0 - h - r2);
    }
    double p_hwe, p_exc;
    site_exact_tests(r0, h, r2, p_hwe, p_exc);
    hwe[i] = p_hwe;
    exchet[i] = p_exc;
}

// ---- genotype posteriors: the allele frequency of a record by EM over its cells' likelihoods, then GP and GQ at it
// (DESIGN.md §8a, "Genotype posteriors").  Every operation is one IEEE double rounded to nearest (intrinsics: no
// contraction), in the order of the statement in tests/test_cohort_posteriors.py.
constexpr int POST_WARPS = 8;                  // records (one per warp) of a thread block
enum : uint32_t { CELL_OUT = 0, CELL_HAP = 1, CELL_DIP = 2 };

// The kind of cell k and its weights w_g = T[PL_g - min PL] (0 beyond the table).  A contributing cell that still has
// NEED_K (its PL was never patched) sets *bad.
__device__ __forceinline__ uint32_t post_weights(const int64_t *__restrict__ pl, const uint8_t *__restrict__ gt,
                                                 const uint8_t *__restrict__ flags, const double *__restrict__ T, size_t k,
                                                 double &w0, double &w1, double &w2, uint32_t *bad) {
    w0 = w1 = w2 = 0.0;
    const uint8_t f = flags[k], g = gt[k];
    if (!(f & SVJG_GT_GENOTYPED) || g == SVJG_GT_NO_CALL) return CELL_OUT;
    if (f & SVJG_GT_NEED_K) atomicOr(bad, 1u);
    const int64_t p0 = pl[3 * k], p1 = pl[3 * k + 1], p2 = pl[3 * k + 2];
    auto wt = [&](int64_t d) { return d > SVJG_POST_PLW_N - 1 ? 0.0 : __ldg(T + d); };
    if (g >= SVJG_GT_HAP_REF) {
        const int64_t m = min(p0, p2);
        w0 = wt(p0 - m);
        w2 = wt(p2 - m);
        return CELL_HAP;
    }
    const int64_t m = min(min(p0, p1), p2);
    w0 = wt(p0 - m);
    w1 = wt(p1 - m);
    w2 = wt(p2 - m);
    return CELL_DIP;
}

// The genotype terms of a cell at f (q = 1 - f; P = q*q, (f*q)*2, f*f): a, b, c and den.  Haploid: a = w0*q, b = 0,
// c = w2*f, den = a + c.
struct PostPriors {
    double f, q, p0, p1, p2;
};
__device__ __forceinline__ PostPriors post_priors(double f) {
    const double q = __dsub_rn(1.0, f);
    return {f, q, __dmul_rn(q, q), __dmul_rn(__dmul_rn(f, q), 2.0), __dmul_rn(f, f)};
}
__device__ __forceinline__ void post_terms(uint32_t kind, double w0, double w1, double w2, const PostPriors &p, double &a,
                                           double &b, double &c, double &den) {
    if (kind == CELL_DIP) {
        a = __dmul_rn(w0, p.p0);
        b = __dmul_rn(w1, p.p1);
        c = __dmul_rn(w2, p.p2);
        den = __dadd_rn(__dadd_rn(a, b), c);
    } else {
        a = __dmul_rn(w0, p.q);
        b = 0.0;
        c = __dmul_rn(w2, p.f);
        den = __dadd_rn(a, c);
    }
}
// expected ALT allele count of a contributing cell: (b + 2c) / den, or c / den for a haploid one
__device__ __forceinline__ double post_e(uint32_t kind, double w0, double w1, double w2, const PostPriors &p) {
    double a, b, c, den;
    post_terms(kind, w0, w1, w2, p, a, b, c, den);
    return kind == CELL_DIP ? __ddiv_rn(__dadd_rn(b, __dmul_rn(c, 2.0)), den) : __ddiv_rn(c, den);
}

// GP of cell k at f̂ into gp[3k..] (haploid: GP1 = 0) and GQ into gq[k]: the largest q <= 99 with err <= T[q], where
// err is the other genotypes' terms over den (T is decreasing, so the q that pass are a prefix: a binary search);
// SVJG_POST_GQ_NONE for a missing call or a cell that does not contribute.
__device__ __forceinline__ void post_cell_out(uint32_t kind, double w0, double w1, double w2, const PostPriors &p,
                                              uint8_t g, const double *__restrict__ T, double *__restrict__ gp,
                                              uint8_t *__restrict__ gq, size_t k) {
    if (kind == CELL_OUT) {
        gp[3 * k] = gp[3 * k + 1] = gp[3 * k + 2] = 0.0;
        gq[k] = SVJG_POST_GQ_NONE;
        return;
    }
    double a, b, c, den;
    post_terms(kind, w0, w1, w2, p, a, b, c, den);
    gp[3 * k] = __ddiv_rn(a, den);
    gp[3 * k + 1] = kind == CELL_DIP ? __ddiv_rn(b, den) : 0.0;
    gp[3 * k + 2] = __ddiv_rn(c, den);
    double other;
    switch (g) {
        case 0: other = __dadd_rn(b, c); break;
        case 1: other = __dadd_rn(a, c); break;
        case 2: other = __dadd_rn(a, b); break;
        case SVJG_GT_HAP_REF: other = c; break;
        case SVJG_GT_HAP_ALT: other = a; break;
        default: gq[k] = SVJG_POST_GQ_NONE; return;   // ./. and . (below -ms, or a tie)
    }
    const double err = __ddiv_rn(other, den);
    uint32_t lo = 0, hi = SVJG_POST_GQ_MAX;            // err <= T[lo] holds (err <= 1 = T[0])
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) / 2;
        if (err <= __ldg(T + mid)) lo = mid;
        else hi = mid - 1;
    }
    gq[k] = uint8_t(lo);
}

__device__ __forceinline__ double warp_sum(double x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x = __dadd_rn(x, __shfl_xor_sync(0xFFFFFFFFu, x, o));
    return x;
}

// One warp per record i of the block the last cohort genotype call left on the device (pl [n][S][3], gt, flags
// [n][S]).  Lane l owns the cells s = l (mod 32).  CPL > 0: S <= 32 CPL, and a lane keeps the weights and kinds of its
// cells in registers.  CPL == 0: any S; the weights are written once into the cell's gp slots and its kind into its
// gq byte, read back (from L2) in every iteration and overwritten by the results at the end.
// Results: af[i] = f̂ (NaN when no cell contributes), iters[i] = EM iterations (0 then), gp [n][S][3], gq [n][S].
template <int CPL>
__global__ void __launch_bounds__(POST_WARPS * 32)
cohort_posterior_kernel(const int64_t *__restrict__ pl, const uint8_t *__restrict__ gt, const uint8_t *__restrict__ flags,
                        uint32_t n, uint32_t S, const double *__restrict__ T, double *__restrict__ af,
                        uint8_t *__restrict__ iters, double *__restrict__ gp, uint8_t *__restrict__ gq,
                        uint32_t *__restrict__ bad) {
    const uint32_t i = blockIdx.x * POST_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= n) return;                                // whole warps leave together
    const size_t row = size_t(i) * S;
    double w[CPL > 0 ? CPL : 1][3];
    uint32_t kind[CPL > 0 ? CPL : 1];
    uint32_t ploidy_sum = 0;
    if constexpr (CPL > 0) {
#pragma unroll
        for (int j = 0; j < CPL; ++j) {
            const uint32_t s = lane + 32 * j;
            kind[j] = CELL_OUT;
            w[j][0] = w[j][1] = w[j][2] = 0.0;
            if (s < S) kind[j] = post_weights(pl, gt, flags, T, row + s, w[j][0], w[j][1], w[j][2], bad);
            ploidy_sum += kind[j];
        }
    } else {
        for (uint32_t s = lane; s < S; s += 32) {
            double w0, w1, w2;
            const uint32_t kd = post_weights(pl, gt, flags, T, row + s, w0, w1, w2, bad);
            gp[3 * (row + s)] = w0;
            gp[3 * (row + s) + 1] = w1;
            gp[3 * (row + s) + 2] = w2;
            gq[row + s] = uint8_t(kd);
            ploidy_sum += kd;
        }
    }
    ploidy_sum = __reduce_add_sync(0xFFFFFFFFu, ploidy_sum);
    double f = __longlong_as_double(0x7FF8000000000000ll);
    uint32_t it = 0;
    if (ploidy_sum) {
        const double A = double(ploidy_sum);
        f = 0.5;
        for (;;) {
            const PostPriors p = post_priors(f);
            double x = 0.0;
            if constexpr (CPL > 0) {
#pragma unroll
                for (int j = 0; j < CPL; ++j)
                    if (kind[j] != CELL_OUT) x = __dadd_rn(x, post_e(kind[j], w[j][0], w[j][1], w[j][2], p));
            } else {
                for (uint32_t s = lane; s < S; s += 32) {
                    const uint32_t kd = gq[row + s];
                    if (kd != CELL_OUT) {
                        const double *wk = gp + 3 * (row + s);
                        x = __dadd_rn(x, post_e(kd, wk[0], wk[1], wk[2], p));
                    }
                }
            }
            const double f_new = __ddiv_rn(warp_sum(x), A);
            ++it;
            const bool done = fabs(__dsub_rn(f_new, f)) <= SVJG_POST_TOL || it == SVJG_POST_MAX_ITERS;
            f = f_new;
            if (done) break;
        }
    }
    if (lane == 0) {
        af[i] = f;
        iters[i] = uint8_t(it);
    }
    const PostPriors p = post_priors(f);
    if constexpr (CPL > 0) {
#pragma unroll
        for (int j = 0; j < CPL; ++j) {
            const uint32_t s = lane + 32 * j;
            if (s < S) post_cell_out(kind[j], w[j][0], w[j][1], w[j][2], p, gt[row + s], T, gp, gq, row + s);
        }
    } else {
        for (uint32_t s = lane; s < S; s += 32) {
            const size_t k = row + s;
            const uint32_t kd = gq[k];
            post_cell_out(kd, gp[3 * k], gp[3 * k + 1], gp[3 * k + 2], p, gt[k], T, gp, gq, k);
        }
    }
}

// The host's PL of the NEED_K cells of the block (svjg_cohort_posteriors' patch) scattered into it, NEED_K cleared
__global__ void cohort_patch_kernel(const uint32_t *__restrict__ cell, const int64_t *__restrict__ patch_pl, uint32_t m,
                                    int64_t *__restrict__ pl, uint8_t *__restrict__ flags) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m) return;
    const size_t c = cell[k];
    pl[3 * c] = patch_pl[3 * size_t(k)];
    pl[3 * c + 1] = patch_pl[3 * size_t(k) + 1];
    pl[3 * c + 2] = patch_pl[3 * size_t(k) + 2];
    flags[c] &= uint8_t(~SVJG_GT_NEED_K);
}

// ---- sample QC and relatedness (DESIGN.md §8a, "Sample QC and relatedness") ----
// Pack: one thread per (sample, QC_PACK_WORDS words of 32 records) of the block the last cohort genotype call left on
// the device.  Bit r of word w of a sample's planes is record 32 w + r of the block: C = diploid called (codes 0-2),
// H = 0/1, A = 1/1; the block's words start at word w0 of the row.  The histogram cell (type row, code) of the thread's
// cells is counted in shared memory (column threadIdx.x: no two threads share a bank) and added to hist [S][5][8]
// with one atomic per non-zero partial; internal row 4 holds the records whose type is not DEL / INS / INV / BND,
// which count in the ALL row only.
constexpr int QC_PACK_THREADS = 128;
constexpr uint32_t QC_PACK_WORDS = 8;
__global__ void __launch_bounds__(QC_PACK_THREADS)
cohort_qc_pack_kernel(const uint8_t *__restrict__ gt, const uint8_t *__restrict__ ty, uint32_t n, uint32_t S,
                      uint32_t *__restrict__ hist, uint32_t *__restrict__ planes, size_t stride, uint32_t w0) {
    __shared__ uint32_t cnt[5 * 8][QC_PACK_THREADS];
    const uint32_t s = blockIdx.x * QC_PACK_THREADS + threadIdx.x;
    if (s >= S) return;                                  // only the thread's own column is used: no barrier
#pragma unroll
    for (int k = 0; k < 5 * 8; ++k) cnt[k][threadIdx.x] = 0;
    const uint32_t n_words = (n + 31) / 32;
    for (uint32_t wlo = blockIdx.y * QC_PACK_WORDS; wlo < n_words; wlo += gridDim.y * QC_PACK_WORDS) {
        const uint32_t whi = min(wlo + QC_PACK_WORDS, n_words);
        for (uint32_t w = wlo; w < whi; ++w) {
            uint32_t C = 0, H = 0, A = 0;
            const uint32_t r0 = 32 * w, r1 = min(r0 + 32, n);
            for (uint32_t r = r0; r < r1; ++r) {
                const uint32_t g = gt[size_t(r) * S + s], t = ty[r] & 0x3F;
                ++cnt[(t <= 3 ? t : 4) * 8 + g][threadIdx.x];
                const uint32_t bit = 1u << (r - r0);
                C |= g <= 2 ? bit : 0u;
                H |= g == 1 ? bit : 0u;
                A |= g == 2 ? bit : 0u;
            }
            if (planes) {
                const size_t o = size_t(s) * stride + w0 + w, plane = size_t(S) * stride;
                planes[o] = C;
                planes[o + plane] = H;
                planes[o + 2 * plane] = A;
            }
        }
    }
    uint32_t *h = hist + size_t(s) * 40;
    for (int g = 0; g < 8; ++g) {
        uint32_t all = 0;
        for (int t = 0; t < 5; ++t) {
            const uint32_t v = cnt[t * 8 + g][threadIdx.x];
            all += v;
            if (t < 4 && v) atomicAdd(h + (1 + t) * 8 + g, v);
        }
        if (all) atomicAdd(h + g, all);
    }
}

// Pairs: the upper triangle of the S x S grid in tiles of PAIR_T x PAIR_T samples, tile (bi, bj) with bi <= bj at
// linear index bj (bj + 1) / 2 + bi.  A K slab of PAIR_KW words of the three planes of both sample ranges is staged in
// shared memory ([side][plane][word][sample]); each thread of a 16 x 16 grid owns the 4 x 4 pairs (i0 + 4 ty + a,
// j0 + 4 tx + b) and keeps five counters per pair.  Per word, with R = C & ~H & ~A (= C ^ H ^ A: H and A are disjoint
// subsets of C): NSV += popc(Ci & Cj), HET1 += popc(Hi & Cj), HET2 += popc(Hj & Ci), HETHET += popc(Hi & Hj),
// IBS0 += popc((Ai & Rj) | (Ri & Aj)).  Pair (i < j) goes to out[5 p], p = i (2 S - i - 1) / 2 + j - i - 1.
constexpr uint32_t PAIR_T = 64;
constexpr uint32_t PAIR_KW = 16;
constexpr int PAIR_THREADS = 256;
__global__ void __launch_bounds__(PAIR_THREADS)
cohort_pair_kernel(const uint32_t *__restrict__ planes, uint32_t S, size_t stride, uint32_t n_slabs,
                   uint32_t *__restrict__ out) {
    __shared__ __align__(16) uint32_t sm[2][3][PAIR_KW][PAIR_T];
    const uint32_t t = blockIdx.x;
    uint32_t bj = uint32_t((sqrt(8.0 * t + 1.0) - 1.0) / 2.0);
    while (bj * (bj + 1) / 2 > t) --bj;
    while ((bj + 1) * (bj + 2) / 2 <= t) ++bj;
    const uint32_t bi = t - bj * (bj + 1) / 2;
    const uint32_t i0 = bi * PAIR_T, j0 = bj * PAIR_T;
    const uint32_t tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const uint32_t lr = threadIdx.x >> 2, lq = threadIdx.x & 3;           // loader: sample lr, words 4 lq .. 4 lq + 3
    const size_t plane = size_t(S) * stride;
    uint32_t cnt[4][4][5];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b)
#pragma unroll
            for (int q = 0; q < 5; ++q) cnt[a][b][q] = 0;
    for (uint32_t slab = 0; slab < n_slabs; ++slab) {
#pragma unroll
        for (int side = 0; side < 2; ++side) {
            const uint32_t row = (side ? j0 : i0) + lr;
#pragma unroll
            for (int p = 0; p < 3; ++p) {
                uint4 v = make_uint4(0, 0, 0, 0);
                if (row < S) v = __ldg(reinterpret_cast<const uint4 *>(planes + p * plane + size_t(row) * stride +
                                                                       size_t(slab) * PAIR_KW + 4 * lq));
                sm[side][p][4 * lq][lr] = v.x;
                sm[side][p][4 * lq + 1][lr] = v.y;
                sm[side][p][4 * lq + 2][lr] = v.z;
                sm[side][p][4 * lq + 3][lr] = v.w;
            }
        }
        __syncthreads();
#pragma unroll 2
        for (uint32_t k = 0; k < PAIR_KW; ++k) {
            const uint4 ci = *reinterpret_cast<const uint4 *>(&sm[0][0][k][4 * ty]);
            const uint4 hi = *reinterpret_cast<const uint4 *>(&sm[0][1][k][4 * ty]);
            const uint4 ai = *reinterpret_cast<const uint4 *>(&sm[0][2][k][4 * ty]);
            const uint4 cj = *reinterpret_cast<const uint4 *>(&sm[1][0][k][4 * tx]);
            const uint4 hj = *reinterpret_cast<const uint4 *>(&sm[1][1][k][4 * tx]);
            const uint4 aj = *reinterpret_cast<const uint4 *>(&sm[1][2][k][4 * tx]);
            const uint32_t Ci[4] = {ci.x, ci.y, ci.z, ci.w}, Hi[4] = {hi.x, hi.y, hi.z, hi.w},
                           Ai[4] = {ai.x, ai.y, ai.z, ai.w};
            const uint32_t Cj[4] = {cj.x, cj.y, cj.z, cj.w}, Hj[4] = {hj.x, hj.y, hj.z, hj.w},
                           Aj[4] = {aj.x, aj.y, aj.z, aj.w};
#pragma unroll
            for (int a = 0; a < 4; ++a) {
                const uint32_t Ri = Ci[a] ^ Hi[a] ^ Ai[a];
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    const uint32_t Rj = Cj[b] ^ Hj[b] ^ Aj[b];
                    cnt[a][b][0] += __popc(Ci[a] & Cj[b]);
                    cnt[a][b][1] += __popc(Hi[a] & Cj[b]);
                    cnt[a][b][2] += __popc(Hj[b] & Ci[a]);
                    cnt[a][b][3] += __popc(Hi[a] & Hj[b]);
                    cnt[a][b][4] += __popc((Ai[a] & Rj) | (Ri & Aj[b]));
                }
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const uint32_t i = i0 + 4 * ty + a;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const uint32_t j = j0 + 4 * tx + b;
            if (i < j && j < S) {
                uint32_t *o = out + 5 * (uint64_t(i) * (2 * uint64_t(S) - i - 1) / 2 + (j - i - 1));
#pragma unroll
                for (int q = 0; q < 5; ++q) o[q] = cnt[a][b][q];
            }
        }
    }
}

// ---- relationship matrix (DESIGN.md §8a, "Relationship matrix and PCA") ----
// Per record: one CTA per plane word w (records 32 w + lane).  Each warp counts the C, H and A bits of its lane's
// record down a stride of the samples, the partials are summed in shared memory, and warp 0 writes the record's
// (u0, u1, u2, v0, v1, v2) to tab [32 n_words][6] and the used-record mask to used[w].  AN = 2 nC, AC = nH + 2 nA; the
// record is used iff 0 < AC < AN and min(AC, AN - AC) / AN >= min_maf; then p = AC / AN, s = 2 p, w = 1 / (s (1 - p)),
// v_g = g - s, u_g = w v_g, each one double operation rounded to nearest.  An unused record's (and a padding bit's)
// entries are 0.
constexpr int GRM_PREP_THREADS = 256;
__global__ void __launch_bounds__(GRM_PREP_THREADS)
cohort_grm_prep_kernel(const uint32_t *__restrict__ planes, uint32_t S, size_t stride, double min_maf,
                       double *__restrict__ tab, uint32_t *__restrict__ used) {
    constexpr int WARPS = GRM_PREP_THREADS / 32;
    __shared__ uint32_t part[3][WARPS][32];
    const uint32_t w = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t plane = size_t(S) * stride;
    uint32_t nc = 0, nh = 0, na = 0;
#pragma unroll 4
    for (uint32_t s = warp; s < S; s += WARPS) {
        const uint32_t *p = planes + size_t(s) * stride + w;
        nc += (__ldg(p) >> lane) & 1;
        nh += (__ldg(p + plane) >> lane) & 1;
        na += (__ldg(p + 2 * plane) >> lane) & 1;
    }
    part[0][warp][lane] = nc;
    part[1][warp][lane] = nh;
    part[2][warp][lane] = na;
    __syncthreads();
    if (warp) return;
    for (int k = 1; k < WARPS; ++k) {
        nc += part[0][k][lane];
        nh += part[1][k][lane];
        na += part[2][k][lane];
    }
    const uint32_t an = 2 * nc, ac = nh + 2 * na;
    const bool use = 0 < ac && ac < an && __ddiv_rn(double(min(ac, an - ac)), double(an)) >= min_maf;
    double t[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    if (use) {
        const double p = __ddiv_rn(double(ac), double(an));
        const double s = __dmul_rn(2.0, p);
        const double wt = __ddiv_rn(1.0, __dmul_rn(s, __dsub_rn(1.0, p)));
#pragma unroll
        for (int g = 0; g < 3; ++g) {
            t[3 + g] = __dsub_rn(double(g), s);
            t[g] = __dmul_rn(wt, t[3 + g]);
        }
    }
    double *o = tab + (size_t(w) * 32 + lane) * 6;
#pragma unroll
    for (int q = 0; q < 6; ++q) o[q] = t[q];
    const uint32_t m = __ballot_sync(0xFFFFFFFFu, use);
    if (lane == 0) used[w] = m;
}

// Pairs: the upper triangle of the S x S grid in tiles of GRM_T x GRM_T samples, tile (bi, bj) with bi <= bj at linear
// index bj (bj + 1) / 2 + bi, as in cohort_pair_kernel.  For each plane word w with a used record, the CTA decodes the
// 32 records of its two sample ranges into shared memory ([side][record][sample]): u_{g_i} on the i side, v_{g_j} on
// the j side, 0.0 for a cell that is not diploid called or a record that is not used (a +-0 term leaves a sum that
// starts at +0.0 unchanged).  Each thread of a 16 x 16 grid owns the 4 x 4 pairs (i0 + 4 ty + a, j0 + tx + 16 b) and
// adds acc = acc + u v record by record in ascending order (__dmul_rn / __dadd_rn: no contraction), with
// N += popc(Ci & U & Cj) per word.  No split over records: every pair sums in record order, so the bits do not depend
// on the tiling.  Pair (i <= j) goes to p = i (2 S - i + 1) / 2 + (j - i): g[p] = acc / N (0.0 when N = 0), n[p] = N.
constexpr uint32_t GRM_T = 64;
constexpr int GRM_THREADS = 256;
__global__ void __launch_bounds__(GRM_THREADS, 2)
cohort_grm_kernel(const uint32_t *__restrict__ planes, uint32_t S, size_t stride, uint32_t n_words,
                  const double *__restrict__ tab, const uint32_t *__restrict__ used, double *__restrict__ g,
                  uint32_t *__restrict__ nout) {
    __shared__ __align__(16) double uv[2][32][GRM_T];
    __shared__ uint32_t cw[2][GRM_T];                                 // C & U of the word, per side and sample
    const uint32_t t = blockIdx.x;
    uint32_t bj = uint32_t((sqrt(8.0 * t + 1.0) - 1.0) / 2.0);
    while (bj * (bj + 1) / 2 > t) --bj;
    while ((bj + 1) * (bj + 2) / 2 <= t) ++bj;
    const uint32_t bi = t - bj * (bj + 1) / 2;
    const uint32_t i0 = bi * GRM_T, j0 = bj * GRM_T;
    const uint32_t tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    // decoder: sample lr of side `side`, records 16 half .. 16 half + 15 of the word
    const uint32_t lr = threadIdx.x & 63, side = (threadIdx.x >> 6) & 1, half = threadIdx.x >> 7;
    const uint32_t row = (side ? j0 : i0) + lr;
    const size_t plane = size_t(S) * stride;
    double acc[4][4];
    uint32_t cnt[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            acc[a][b] = 0.0;
            cnt[a][b] = 0;
        }
    for (uint32_t w = 0; w < n_words; ++w) {
        const uint32_t U = __ldg(used + w);
        if (U == 0) continue;                                           // the same for the whole CTA
        uint32_t Cw = 0, Hw = 0, Aw = 0;
        if (row < S) {
            const uint32_t *p = planes + size_t(row) * stride + w;
            Cw = __ldg(p) & U;
            Hw = __ldg(p + plane);
            Aw = __ldg(p + 2 * plane);
        }
        if (half == 0) cw[side][lr] = Cw;
        const double *tw = tab + size_t(w) * 32 * 6 + 3 * side;
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            const uint32_t r = 16 * half + k, bit = 1u << r;
            double x = 0.0;
            if (Cw & bit) x = __ldg(tw + r * 6 + ((Hw & bit) ? 1 : (Aw & bit) ? 2 : 0));
            uv[side][r][lr] = x;
        }
        __syncthreads();
        uint32_t Ci[4], Cj[4];
#pragma unroll
        for (int a = 0; a < 4; ++a) Ci[a] = cw[0][4 * ty + a];
#pragma unroll
        for (int b = 0; b < 4; ++b) Cj[b] = cw[1][tx + 16 * b];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) cnt[a][b] += __popc(Ci[a] & Cj[b]);
#pragma unroll 4
        for (int k = 0; k < 32; ++k) {
            const double2 u01 = *reinterpret_cast<const double2 *>(&uv[0][k][4 * ty]);
            const double2 u23 = *reinterpret_cast<const double2 *>(&uv[0][k][4 * ty + 2]);
            const double ui[4] = {u01.x, u01.y, u23.x, u23.y};
            double vj[4];
#pragma unroll
            for (int b = 0; b < 4; ++b) vj[b] = uv[1][k][tx + 16 * b];
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) acc[a][b] = __dadd_rn(acc[a][b], __dmul_rn(ui[a], vj[b]));
        }
        __syncthreads();
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const uint32_t i = i0 + 4 * ty + a;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const uint32_t j = j0 + tx + 16 * b;
            if (i <= j && j < S) {
                const uint64_t p = uint64_t(i) * (2 * uint64_t(S) - i + 1) / 2 + (j - i);
                nout[p] = cnt[a][b];
                g[p] = cnt[a][b] ? __ddiv_rn(acc[a][b], double(cnt[a][b])) : 0.0;
            }
        }
    }
}

}  // namespace

extern "C" int svjg_genotype_device(const uint32_t *d_counts, const uint32_t *d_sv_index, const uint8_t *d_svtype,
                                    uint32_t n, int64_t min_support, double log10_1me, double log10_e,
                                    double log10_half, const double *d_lut, uint32_t lut_nmax,
                                    const double *d_k_override, int64_t *d_pl, uint8_t *d_gt, uint32_t *d_ad2,
                                    uint8_t *d_flags, void *stream) {
    if (n == 0) return SVJG_OK;
    if (!d_counts || !d_sv_index || !d_svtype || !d_lut || !d_pl || !d_gt || !d_ad2 || !d_flags)
        return svjg::set_error(SVJG_E_ARG, "svjg_genotype_device: NULL argument");
    if (!(log10_1me == log10_1me) || !(log10_e == log10_e) || !(log10_half == log10_half))
        return svjg::set_error(SVJG_E_ARG, "svjg_genotype_device: NaN constant");
    int threads = 128;
    int blocks = int((uint64_t(n) + threads - 1) / threads);
    genotype_kernel<false><<<blocks, threads, 0, (cudaStream_t)stream>>>(d_counts, Xchg{}, d_sv_index, d_svtype, n, min_support,
                                                                         log10_1me, log10_e, log10_half, d_lut, lut_nmax,
                                                                         d_k_override, d_pl, d_gt, d_ad2, d_flags);
    SVJG_CUDA(cudaGetLastError());
    return SVJG_OK;
}

// Same from host arrays: device buffers are this call's own (the stand-alone predict-genotype
// front-end needs nothing else from the GPU, so it does not have to load a tensor library).
extern "C" int svjg_genotype_host(const uint32_t *counts, uint32_t num_counts, const uint32_t *sv_index, const uint8_t *svtype,
                                  uint32_t n, int64_t min_support, double log10_1me, double log10_e, double log10_half,
                                  const double *lut, uint32_t lut_nmax, const double *k_override, int64_t *pl, uint8_t *gt,
                                  uint32_t *ad2, uint8_t *flags) {
    if (n == 0) return SVJG_OK;
    if (!sv_index || !svtype || !lut || !pl || !gt || !ad2 || !flags || (num_counts && !counts))
        return svjg::set_error(SVJG_E_ARG, "svjg_genotype_host: NULL argument");
    const size_t n_lut = size_t(lut_nmax + 1) * (lut_nmax + 2) / 2;
    const size_t b_cnt = std::max<size_t>(8, size_t(num_counts) * 8), b_idx = size_t(n) * 4, b_ty = n, b_lut = n_lut * 8,
                 b_k = k_override ? size_t(n) * 8 : 0, b_pl = size_t(n) * 24, b_gt = n, b_ad = size_t(n) * 8, b_fl = n;
    auto up = [](size_t x) { return (x + 255) & ~size_t(255); };
    const size_t o_idx = up(b_cnt), o_ty = o_idx + up(b_idx), o_lut = o_ty + up(b_ty), o_k = o_lut + up(b_lut),
                 o_pl = o_k + up(b_k), o_gt = o_pl + up(b_pl), o_ad = o_gt + up(b_gt), o_fl = o_ad + up(b_ad),
                 total = o_fl + up(b_fl);
    // a stream of the call's own and stream-ordered memory: nothing here waits for other work on the device
    // (the JSON text of the same file may be on its way back, svjg_filter_json_finish)
    cudaStream_t st = nullptr;
    SVJG_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    uint8_t *d = nullptr;
    cudaError_t e = cudaMallocAsync(reinterpret_cast<void **>(&d), total, st);
    if (e != cudaSuccess) {
        cudaStreamDestroy(st);
        return svjg::cuda_fail(int(e), "svjg_genotype_host: device memory");
    }
    int rc = SVJG_OK;
    auto h2d = [&](size_t off, const void *src, size_t bytes) {
        if (e == cudaSuccess && bytes) e = cudaMemcpyAsync(d + off, src, bytes, cudaMemcpyHostToDevice, st);
    };
    if (num_counts) h2d(0, counts, size_t(num_counts) * 8);
    h2d(o_idx, sv_index, b_idx);
    h2d(o_ty, svtype, b_ty);
    h2d(o_lut, lut, b_lut);
    h2d(o_k, k_override, b_k);
    if (e == cudaSuccess)
        rc = svjg_genotype_device(reinterpret_cast<const uint32_t *>(d), reinterpret_cast<const uint32_t *>(d + o_idx), d + o_ty, n,
                                  min_support, log10_1me, log10_e, log10_half, reinterpret_cast<const double *>(d + o_lut),
                                  lut_nmax, k_override ? reinterpret_cast<const double *>(d + o_k) : nullptr,
                                  reinterpret_cast<int64_t *>(d + o_pl), d + o_gt, reinterpret_cast<uint32_t *>(d + o_ad),
                                  d + o_fl, st);
    auto d2h = [&](void *dst, size_t off, size_t bytes) {
        if (e == cudaSuccess && rc == SVJG_OK) e = cudaMemcpyAsync(dst, d + off, bytes, cudaMemcpyDeviceToHost, st);
    };
    d2h(pl, o_pl, b_pl);
    d2h(gt, o_gt, b_gt);
    d2h(ad2, o_ad, b_ad);
    d2h(flags, o_fl, b_fl);
    cudaFreeAsync(d, st);
    const cudaError_t es = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = es;
    cudaStreamDestroy(st);
    if (e != cudaSuccess) return svjg::cuda_fail(int(e), "svjg_genotype_host");
    return rc;
}

// ---------------------------------------------------------------------------
// cohort: one block of records genotyped in every sample
// ---------------------------------------------------------------------------
extern "C" int svjg_cohort_set_ploidy(svjg_cohort *c, uint32_t n_classes, uint32_t n_sexes, const uint8_t *table,
                                      const uint8_t *sample_sex) {
    if (!c || !table || !sample_sex) return svjg::set_error(SVJG_E_ARG, "svjg_cohort_set_ploidy: NULL argument");
    if (n_classes == 0 || n_classes > SVJG_PLOIDY_MAX_CLASSES || n_sexes == 0 || n_sexes > SVJG_PLOIDY_MAX_SEXES)
        return svjg::set_error(SVJG_E_ARG, "svjg_cohort_set_ploidy: 1 to 255 classes and 1 to 64 sexes");
    const size_t n_tab = size_t(n_classes) * n_sexes;
    for (size_t k = 0; k < n_tab; ++k)
        if (table[k] > 2) return svjg::set_error(SVJG_E_ARG, "svjg_cohort_set_ploidy: a ploidy other than 0, 1 or 2");
    for (uint32_t s = 0; s < c->n_samples; ++s)
        if (sample_sex[s] >= n_sexes) return svjg::set_error(SVJG_E_ARG, "svjg_cohort_set_ploidy: sample sex out of range");
    SVJG_CUDA(cudaSetDevice(c->t->device));
    if (c->d_ploidy) SVJG_CUDA(cudaFree(c->d_ploidy));
    c->d_ploidy = nullptr;
    c->n_classes = c->n_sexes = 0;
    // [n_classes][n_sexes] table, then the sex of every sample
    SVJG_CUDA(cudaMalloc(&c->d_ploidy, n_tab + c->n_samples));
    SVJG_CUDA(cudaMemcpy(c->d_ploidy, table, n_tab, cudaMemcpyHostToDevice));
    SVJG_CUDA(cudaMemcpy(c->d_ploidy + n_tab, sample_sex, c->n_samples, cudaMemcpyHostToDevice));
    c->n_classes = n_classes;
    c->n_sexes = n_sexes;
    return SVJG_OK;
}

namespace {
// svjg_cohort_genotype (rclass == nullptr: every cell diploid) and svjg_cohort_genotype_ploidy
int cohort_genotype(const char *fn, svjg_cohort *c, const uint32_t *sv_index, const uint8_t *svtype, const uint8_t *rclass,
                    uint32_t n, int64_t min_support, double log10_1me, double log10_e, double log10_half, const double *lut,
                    uint32_t lut_nmax, int64_t *pl, uint8_t *gt, uint32_t *ad2, uint8_t *flags) {
    const std::string f = fn;
    if (!c) return svjg::set_error(SVJG_E_ARG, f + ": NULL cohort");
    c->blk_n = 0;                          // set again once this block's cells are complete
    c->blk_qc = false;
    if (n == 0) return SVJG_OK;
    if (!sv_index || !svtype || !lut || !pl || !gt || !ad2 || !flags)
        return svjg::set_error(SVJG_E_ARG, f + ": NULL argument");
    if (!(log10_1me == log10_1me) || !(log10_e == log10_e) || !(log10_half == log10_half))
        return svjg::set_error(SVJG_E_ARG, f + ": NaN constant");
    const uint64_t cells = uint64_t(n) * c->n_samples;
    if (cells >= 0xFFFFFFFFull) return svjg::set_error(SVJG_E_ARG, f + ": block of more than 2^32 cells");
    for (uint32_t i = 0; i < n; ++i)
        if (sv_index[i] != 0xFFFFFFFFu && sv_index[i] >= c->num_sv)
            return svjg::set_error(SVJG_E_ARG, f + ": sv_index out of range");
    if (rclass) {
        if (!c->d_ploidy) return svjg::set_error(SVJG_E_ARG, f + ": no ploidy table (svjg_cohort_set_ploidy)");
        for (uint32_t i = 0; i < n; ++i)
            if (rclass[i] >= c->n_classes) return svjg::set_error(SVJG_E_ARG, f + ": record class out of range");
    }
    SVJG_CUDA(cudaSetDevice(c->t->device));
    // the LUT is uploaded again only when its contents change
    const size_t n_lut = size_t(lut_nmax + 1) * (lut_nmax + 2) / 2;
    if (c->lut.size() != n_lut || memcmp(c->lut.data(), lut, n_lut * 8) != 0) {
        if (c->d_lut) SVJG_CUDA(cudaFree(c->d_lut));
        c->d_lut = nullptr;
        c->lut.clear();
        SVJG_CUDA(cudaMalloc(&c->d_lut, n_lut * 8));
        SVJG_CUDA(cudaMemcpy(c->d_lut, lut, n_lut * 8, cudaMemcpyHostToDevice));
        c->lut.assign(lut, lut + n_lut);
    }
    auto up = [](size_t x) { return (x + 255) & ~size_t(255); };
    const size_t b_idx = size_t(n) * 4, b_ty = n, b_cls = rclass ? n : 0, b_pl = cells * 24, b_gt = cells, b_ad = cells * 8,
                 b_fl = cells;
    const size_t o_ty = up(b_idx), o_cls = o_ty + up(b_ty), o_pl = o_cls + up(b_cls), o_gt = o_pl + up(b_pl),
                 o_ad = o_gt + up(b_gt), o_fl = o_ad + up(b_ad), total = o_fl + up(b_fl);
    if (c->blk_cap < total) {
        if (c->d_blk) SVJG_CUDA(cudaFree(c->d_blk));
        c->d_blk = nullptr;
        c->blk_cap = 0;
        SVJG_CUDA(cudaMalloc(&c->d_blk, total));
        c->blk_cap = total;
    }
    uint8_t *d = c->d_blk;
    cudaStream_t st = c->stream;
    SVJG_CUDA(cudaMemcpyAsync(d, sv_index, b_idx, cudaMemcpyHostToDevice, st));
    SVJG_CUDA(cudaMemcpyAsync(d + o_ty, svtype, b_ty, cudaMemcpyHostToDevice, st));
    if (rclass) SVJG_CUDA(cudaMemcpyAsync(d + o_cls, rclass, b_cls, cudaMemcpyHostToDevice, st));
    const int threads = 128;
    const uint32_t blocks = uint32_t((cells + threads - 1) / threads);
    auto kernel = rclass ? genotype_cohort_kernel<true> : genotype_cohort_kernel<false>;
    const uint8_t *d_tab = rclass ? c->d_ploidy : nullptr;
    kernel<<<blocks, threads, 0, st>>>(c->d_counts, c->num_sv, c->n_samples, reinterpret_cast<const uint32_t *>(d), d + o_ty,
                                       uint32_t(cells), min_support, log10_1me, log10_e, log10_half, c->d_lut, lut_nmax,
                                       reinterpret_cast<int64_t *>(d + o_pl), d + o_gt, reinterpret_cast<uint32_t *>(d + o_ad),
                                       d + o_fl, rclass ? d + o_cls : nullptr,
                                       d_tab ? d_tab + size_t(c->n_classes) * c->n_sexes : nullptr, d_tab, c->n_sexes);
    SVJG_CUDA(cudaGetLastError());
    SVJG_CUDA(cudaMemcpyAsync(pl, d + o_pl, b_pl, cudaMemcpyDeviceToHost, st));
    SVJG_CUDA(cudaMemcpyAsync(gt, d + o_gt, b_gt, cudaMemcpyDeviceToHost, st));
    SVJG_CUDA(cudaMemcpyAsync(ad2, d + o_ad, b_ad, cudaMemcpyDeviceToHost, st));
    SVJG_CUDA(cudaMemcpyAsync(flags, d + o_fl, b_fl, cudaMemcpyDeviceToHost, st));
    SVJG_CUDA(cudaStreamSynchronize(st));
    c->blk_n = n;
    c->blk_gt = o_gt;
    c->blk_pl = o_pl;
    c->blk_fl = o_fl;
    c->blk_ty = o_ty;
    return SVJG_OK;
}

// Site statistics of the block of the last genotype call, from its gt codes where the kernel left them on the device:
// 32 B (40 B with ploidy) per record come back, not the cells.
int cohort_site_stats(const char *fn, bool ploidy, svjg_cohort *c, uint32_t n, uint32_t *gcount, double *hwe, double *exchet) {
    const std::string f = fn;
    if (!c) return svjg::set_error(SVJG_E_ARG, f + ": NULL cohort");
    if (n != c->blk_n)
        return svjg::set_error(SVJG_E_ARG, f + ": n is not the record count of the last svjg_cohort_genotype call");
    if (n == 0) return SVJG_OK;
    if (!gcount || !hwe || !exchet) return svjg::set_error(SVJG_E_ARG, f + ": NULL argument");
    // every D and E of the exact tests must be exact in a double
    const uint64_t s1 = uint64_t(c->n_samples) + 1;
    if (s1 >= (1ull << 26) || 4 * s1 * s1 >= (1ull << 53))
        return svjg::set_error(SVJG_E_ARG, f + ": 4 (S + 1)^2 must be below 2^53");
    SVJG_CUDA(cudaSetDevice(c->t->device));
    auto up = [](size_t x) { return (x + 255) & ~size_t(255); };
    const size_t b_cnt = size_t(n) * (ploidy ? 24 : 16), b_p = size_t(n) * 8, o_hwe = up(b_cnt), o_exc = o_hwe + up(b_p),
                 total = o_exc + up(b_p);
    if (c->site_cap < total) {
        if (c->d_site) SVJG_CUDA(cudaFree(c->d_site));
        c->d_site = nullptr;
        c->site_cap = 0;
        SVJG_CUDA(cudaMalloc(&c->d_site, total));
        c->site_cap = total;
    }
    uint8_t *d = c->d_site;
    cudaStream_t st = c->stream;
    const uint32_t blocks = uint32_t((uint64_t(n) + SITE_THREADS - 1) / SITE_THREADS);
    auto kernel = ploidy ? cohort_site_stats_kernel<true> : cohort_site_stats_kernel<false>;
    kernel<<<blocks, SITE_THREADS, 0, st>>>(c->d_blk + c->blk_gt, n, c->n_samples, reinterpret_cast<uint32_t *>(d),
                                            reinterpret_cast<double *>(d + o_hwe), reinterpret_cast<double *>(d + o_exc));
    SVJG_CUDA(cudaGetLastError());
    SVJG_CUDA(cudaMemcpyAsync(gcount, d, b_cnt, cudaMemcpyDeviceToHost, st));
    SVJG_CUDA(cudaMemcpyAsync(hwe, d + o_hwe, b_p, cudaMemcpyDeviceToHost, st));
    SVJG_CUDA(cudaMemcpyAsync(exchet, d + o_exc, b_p, cudaMemcpyDeviceToHost, st));
    SVJG_CUDA(cudaStreamSynchronize(st));
    return SVJG_OK;
}
}  // namespace

extern "C" int svjg_cohort_genotype(svjg_cohort *c, const uint32_t *sv_index, const uint8_t *svtype, uint32_t n,
                                    int64_t min_support, double log10_1me, double log10_e, double log10_half,
                                    const double *lut, uint32_t lut_nmax, int64_t *pl, uint8_t *gt, uint32_t *ad2,
                                    uint8_t *flags) {
    return cohort_genotype("svjg_cohort_genotype", c, sv_index, svtype, nullptr, n, min_support, log10_1me, log10_e,
                           log10_half, lut, lut_nmax, pl, gt, ad2, flags);
}

extern "C" int svjg_cohort_genotype_ploidy(svjg_cohort *c, const uint32_t *sv_index, const uint8_t *svtype,
                                           const uint8_t *rclass, uint32_t n, int64_t min_support, double log10_1me,
                                           double log10_e, double log10_half, const double *lut, uint32_t lut_nmax,
                                           int64_t *pl, uint8_t *gt, uint32_t *ad2, uint8_t *flags) {
    if (n && !rclass) return svjg::set_error(SVJG_E_ARG, "svjg_cohort_genotype_ploidy: NULL argument");
    return cohort_genotype("svjg_cohort_genotype_ploidy", c, sv_index, svtype, rclass, n, min_support, log10_1me, log10_e,
                           log10_half, lut, lut_nmax, pl, gt, ad2, flags);
}

extern "C" int svjg_cohort_site_stats(svjg_cohort *c, uint32_t n, uint32_t *gcount, double *hwe, double *exchet) {
    return cohort_site_stats("svjg_cohort_site_stats", false, c, n, gcount, hwe, exchet);
}

extern "C" int svjg_cohort_site_stats_ploidy(svjg_cohort *c, uint32_t n, uint32_t *gcount, double *hwe, double *exchet) {
    return cohort_site_stats("svjg_cohort_site_stats_ploidy", true, c, n, gcount, hwe, exchet);
}

// Genotype posteriors of the block of the last genotype call, from its pl / gt / flags where that call left them on the
// device: the host's PLs of the NEED_K cells go in first, then one warp per record runs the EM and writes GP and GQ.
extern "C" int svjg_cohort_posteriors(svjg_cohort *c, uint32_t n, uint32_t n_patch, const uint32_t *patch_cell,
                                      const int64_t *patch_pl, const double *plw, uint32_t plw_n, double *af, double *gp,
                                      uint8_t *gq, uint8_t *iters) {
    const std::string f = "svjg_cohort_posteriors";
    if (!c) return svjg::set_error(SVJG_E_ARG, f + ": NULL cohort");
    if (n != c->blk_n)
        return svjg::set_error(SVJG_E_ARG, f + ": n is not the record count of the last svjg_cohort_genotype call");
    if (n == 0) return SVJG_OK;
    if (!plw || !af || !gp || !gq || (n_patch && (!patch_cell || !patch_pl)))
        return svjg::set_error(SVJG_E_ARG, f + ": NULL argument");
    if (plw_n != SVJG_POST_PLW_N) return svjg::set_error(SVJG_E_ARG, f + ": the weight table must have SVJG_POST_PLW_N entries");
    const uint64_t cells = uint64_t(n) * c->n_samples;
    for (uint32_t k = 0; k < n_patch; ++k)
        if (patch_cell[k] >= cells) return svjg::set_error(SVJG_E_ARG, f + ": patch cell out of range");
    SVJG_CUDA(cudaSetDevice(c->t->device));
    cudaStream_t st = c->stream;
    // the table is uploaded again only when its contents change
    if (c->plw.size() != plw_n || memcmp(c->plw.data(), plw, size_t(plw_n) * 8) != 0) {
        if (c->d_plw) SVJG_CUDA(cudaFree(c->d_plw));
        c->d_plw = nullptr;
        c->plw.clear();
        SVJG_CUDA(cudaMalloc(&c->d_plw, size_t(plw_n) * 8));
        SVJG_CUDA(cudaMemcpy(c->d_plw, plw, size_t(plw_n) * 8, cudaMemcpyHostToDevice));
        c->plw.assign(plw, plw + plw_n);
    }
    auto up = [](size_t x) { return (x + 255) & ~size_t(255); };
    const size_t b_pc = size_t(n_patch) * 4, b_pp = size_t(n_patch) * 24, b_af = size_t(n) * 8, b_it = n,
                 b_gp = cells * 24, b_gq = cells;
    const size_t o_pp = up(b_pc), o_af = o_pp + up(b_pp), o_it = o_af + up(b_af), o_gp = o_it + up(b_it),
                 o_gq = o_gp + up(b_gp), o_bad = o_gq + up(b_gq), total = o_bad + 256;
    if (c->post_cap < total) {
        if (c->d_post) SVJG_CUDA(cudaFree(c->d_post));
        c->d_post = nullptr;
        c->post_cap = 0;
        SVJG_CUDA(cudaMalloc(&c->d_post, total));
        c->post_cap = total;
    }
    uint8_t *d = c->d_post, *blk = c->d_blk;
    int64_t *d_pl = reinterpret_cast<int64_t *>(blk + c->blk_pl);
    uint32_t *d_bad = reinterpret_cast<uint32_t *>(d + o_bad);
    if (n_patch) {
        SVJG_CUDA(cudaMemcpyAsync(d, patch_cell, b_pc, cudaMemcpyHostToDevice, st));
        SVJG_CUDA(cudaMemcpyAsync(d + o_pp, patch_pl, b_pp, cudaMemcpyHostToDevice, st));
        cohort_patch_kernel<<<(n_patch + 255) / 256, 256, 0, st>>>(reinterpret_cast<const uint32_t *>(d),
                                                                  reinterpret_cast<const int64_t *>(d + o_pp), n_patch,
                                                                  d_pl, blk + c->blk_fl);
        SVJG_CUDA(cudaGetLastError());
    }
    SVJG_CUDA(cudaMemsetAsync(d_bad, 0, 4, st));
    // weights in registers while a lane has at most 4 cells, else written once into the gp slots and read from L2
    const uint32_t S = c->n_samples;
    auto kernel = S <= 32 ? cohort_posterior_kernel<1> : S <= 64 ? cohort_posterior_kernel<2>
                : S <= 128 ? cohort_posterior_kernel<4> : cohort_posterior_kernel<0>;
    kernel<<<(n + POST_WARPS - 1) / POST_WARPS, POST_WARPS * 32, 0, st>>>(
        d_pl, blk + c->blk_gt, blk + c->blk_fl, n, S, c->d_plw, reinterpret_cast<double *>(d + o_af), d + o_it,
        reinterpret_cast<double *>(d + o_gp), d + o_gq, d_bad);
    SVJG_CUDA(cudaGetLastError());
    uint32_t bad = 0;
    SVJG_CUDA(cudaMemcpyAsync(af, d + o_af, b_af, cudaMemcpyDeviceToHost, st));
    if (iters) SVJG_CUDA(cudaMemcpyAsync(iters, d + o_it, b_it, cudaMemcpyDeviceToHost, st));
    SVJG_CUDA(cudaMemcpyAsync(gp, d + o_gp, b_gp, cudaMemcpyDeviceToHost, st));
    SVJG_CUDA(cudaMemcpyAsync(gq, d + o_gq, b_gq, cudaMemcpyDeviceToHost, st));
    SVJG_CUDA(cudaMemcpyAsync(&bad, d_bad, 4, cudaMemcpyDeviceToHost, st));
    SVJG_CUDA(cudaStreamSynchronize(st));
    if (bad) return svjg::set_error(SVJG_E_ARG, f + ": a contributing cell still has SVJG_GT_NEED_K (no PL patched in)");
    return SVJG_OK;
}

// Sample QC and relatedness: resident histogram and bit planes, filled block by block, read once at the end.
extern "C" int svjg_cohort_qc_begin(svjg_cohort *c, uint32_t n_words, int want_pairs) {
    const std::string f = "svjg_cohort_qc_begin";
    if (!c) return svjg::set_error(SVJG_E_ARG, f + ": NULL cohort");
    if (want_pairs && c->n_samples > SVJG_QC_MAX_PAIR_SAMPLES)
        return svjg::set_error(SVJG_E_ARG, f + ": relatedness takes at most SVJG_QC_MAX_PAIR_SAMPLES samples");
    SVJG_CUDA(cudaSetDevice(c->t->device));
    if (c->d_qc) SVJG_CUDA(cudaFree(c->d_qc));
    c->d_qc = nullptr;
    c->qc_on = false;
    const size_t S = c->n_samples, stride = (size_t(n_words) + PAIR_KW - 1) / PAIR_KW * PAIR_KW;
    const size_t words = S * 40 + (want_pairs ? 3 * S * stride : 0);
    SVJG_CUDA(cudaMalloc(&c->d_qc, words * 4));
    SVJG_CUDA(cudaMemset(c->d_qc, 0, words * 4));
    c->qc_words = n_words;
    c->qc_used = 0;
    c->qc_stride = stride;
    c->qc_pairs = want_pairs != 0;
    c->qc_on = true;
    return SVJG_OK;
}

extern "C" int svjg_cohort_qc_add(svjg_cohort *c, uint32_t n) {
    const std::string f = "svjg_cohort_qc_add";
    if (!c) return svjg::set_error(SVJG_E_ARG, f + ": NULL cohort");
    if (!c->qc_on) return svjg::set_error(SVJG_E_ARG, f + ": no svjg_cohort_qc_begin");
    if (n != c->blk_n)
        return svjg::set_error(SVJG_E_ARG, f + ": n is not the record count of the last svjg_cohort_genotype call");
    if (n == 0) return SVJG_OK;
    if (c->blk_qc) return svjg::set_error(SVJG_E_ARG, f + ": the block of the last genotype call was added already");
    const uint32_t words = (n + 31) / 32;
    if (uint64_t(c->qc_used) + words > c->qc_words)
        return svjg::set_error(SVJG_E_ARG, f + ": more words than svjg_cohort_qc_begin's n_words");
    SVJG_CUDA(cudaSetDevice(c->t->device));
    const uint32_t S = c->n_samples;
    const dim3 grid((S + QC_PACK_THREADS - 1) / QC_PACK_THREADS, std::min<uint32_t>((words + QC_PACK_WORDS - 1) / QC_PACK_WORDS, 65535));
    cohort_qc_pack_kernel<<<grid, QC_PACK_THREADS, 0, c->stream>>>(c->d_blk + c->blk_gt, c->d_blk + c->blk_ty, n, S, c->d_qc,
                                                                   c->qc_pairs ? c->d_qc + size_t(S) * 40 : nullptr,
                                                                   c->qc_stride, c->qc_used);
    SVJG_CUDA(cudaGetLastError());
    c->qc_used += words;
    c->blk_qc = true;
    return SVJG_OK;
}

extern "C" int svjg_cohort_qc_sample_counts(svjg_cohort *c, uint32_t *out) {
    if (!c || !out) return svjg::set_error(SVJG_E_ARG, "svjg_cohort_qc_sample_counts: NULL argument");
    if (!c->qc_on) return svjg::set_error(SVJG_E_ARG, "svjg_cohort_qc_sample_counts: no svjg_cohort_qc_begin");
    SVJG_CUDA(cudaSetDevice(c->t->device));
    SVJG_CUDA(cudaMemcpyAsync(out, c->d_qc, size_t(c->n_samples) * 40 * 4, cudaMemcpyDeviceToHost, c->stream));
    SVJG_CUDA(cudaStreamSynchronize(c->stream));
    return SVJG_OK;
}

extern "C" int svjg_cohort_qc_planes(svjg_cohort *c, uint32_t *out) {
    const std::string f = "svjg_cohort_qc_planes";
    if (!c || !out) return svjg::set_error(SVJG_E_ARG, f + ": NULL argument");
    if (!c->qc_on || !c->qc_pairs) return svjg::set_error(SVJG_E_ARG, f + ": no svjg_cohort_qc_begin with want_pairs");
    if (c->qc_words == 0) return SVJG_OK;
    SVJG_CUDA(cudaSetDevice(c->t->device));
    SVJG_CUDA(cudaMemcpy2DAsync(out, size_t(c->qc_words) * 4, c->d_qc + size_t(c->n_samples) * 40, c->qc_stride * 4,
                                size_t(c->qc_words) * 4, 3 * size_t(c->n_samples), cudaMemcpyDeviceToHost, c->stream));
    SVJG_CUDA(cudaStreamSynchronize(c->stream));
    return SVJG_OK;
}

extern "C" int svjg_cohort_relatedness(svjg_cohort *c, uint32_t *out) {
    const std::string f = "svjg_cohort_relatedness";
    if (!c) return svjg::set_error(SVJG_E_ARG, f + ": NULL cohort");
    if (!c->qc_on || !c->qc_pairs) return svjg::set_error(SVJG_E_ARG, f + ": no svjg_cohort_qc_begin with want_pairs");
    const uint64_t S = c->n_samples, n_pairs = S * (S - 1) / 2;
    if (n_pairs == 0) return SVJG_OK;
    if (!out) return svjg::set_error(SVJG_E_ARG, f + ": NULL argument");
    SVJG_CUDA(cudaSetDevice(c->t->device));
    cudaStream_t st = c->stream;
    uint32_t *d_out = nullptr;
    SVJG_CUDA(cudaMallocAsync(reinterpret_cast<void **>(&d_out), n_pairs * 20, st));
    const uint64_t tiles = (S + PAIR_T - 1) / PAIR_T;
    const uint32_t n_slabs = uint32_t((uint64_t(c->qc_used) + PAIR_KW - 1) / PAIR_KW);
    cudaError_t e = cudaSuccess;
    if (n_slabs == 0) e = cudaMemsetAsync(d_out, 0, n_pairs * 20, st);
    else cohort_pair_kernel<<<uint32_t(tiles * (tiles + 1) / 2), PAIR_THREADS, 0, st>>>(c->d_qc + S * 40, uint32_t(S),
                                                                                         c->qc_stride, n_slabs, d_out);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_out, n_pairs * 20, cudaMemcpyDeviceToHost, st);
    cudaFreeAsync(d_out, st);
    const cudaError_t es = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = es;
    if (e != cudaSuccess) return svjg::cuda_fail(int(e), "svjg_cohort_relatedness");
    return SVJG_OK;
}

// Relationship matrix over the resident planes: the per-record table, then the pair tiles; the planes are only read.
extern "C" int svjg_cohort_grm(svjg_cohort *c, double min_maf, double *grm, uint32_t *n) {
    const std::string f = "svjg_cohort_grm";
    if (!c) return svjg::set_error(SVJG_E_ARG, f + ": NULL cohort");
    if (!c->qc_on || !c->qc_pairs) return svjg::set_error(SVJG_E_ARG, f + ": no svjg_cohort_qc_begin with want_pairs");
    if (!(min_maf >= 0.0 && min_maf <= 0.5)) return svjg::set_error(SVJG_E_ARG, f + ": min_maf must be in [0, 0.5]");
    const uint64_t S = c->n_samples, n_pairs = S * (S + 1) / 2;
    if (n_pairs == 0) return SVJG_OK;
    if (!grm || !n) return svjg::set_error(SVJG_E_ARG, f + ": NULL argument");
    SVJG_CUDA(cudaSetDevice(c->t->device));
    cudaStream_t st = c->stream;
    const uint64_t n_words = c->qc_used;
    // one allocation: G [n_pairs] f64, the table [32 n_words][6] f64, N [n_pairs] u32, the mask [n_words] u32
    const size_t o_tab = n_pairs * 8, o_n = o_tab + n_words * 32 * 6 * 8, o_used = o_n + n_pairs * 4;
    char *d = nullptr;
    SVJG_CUDA(cudaMallocAsync(reinterpret_cast<void **>(&d), o_used + n_words * 4, st));
    double *d_g = reinterpret_cast<double *>(d), *d_tab = reinterpret_cast<double *>(d + o_tab);
    uint32_t *d_n = reinterpret_cast<uint32_t *>(d + o_n), *d_used = reinterpret_cast<uint32_t *>(d + o_used);
    const uint32_t *planes = c->d_qc + S * 40;
    const uint64_t tiles = (S + GRM_T - 1) / GRM_T;
    cudaError_t e = cudaSuccess;
    if (n_words == 0) {
        e = cudaMemsetAsync(d, 0, o_used, st);
    } else {
        cohort_grm_prep_kernel<<<uint32_t(n_words), GRM_PREP_THREADS, 0, st>>>(planes, uint32_t(S), c->qc_stride, min_maf,
                                                                                d_tab, d_used);
        e = cudaGetLastError();
        if (e == cudaSuccess)
            cohort_grm_kernel<<<uint32_t(tiles * (tiles + 1) / 2), GRM_THREADS, 0, st>>>(
                planes, uint32_t(S), c->qc_stride, uint32_t(n_words), d_tab, d_used, d_g, d_n);
    }
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(grm, d_g, n_pairs * 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(n, d_n, n_pairs * 4, cudaMemcpyDeviceToHost, st);
    cudaFreeAsync(d, st);
    const cudaError_t es = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = es;
    if (e != cudaSuccess) return svjg::cuda_fail(int(e), "svjg_cohort_grm");
    return SVJG_OK;
}

// ---------------------------------------------------------------------------
// counter exchange between the ranks of one node (one process per GPU)
// ---------------------------------------------------------------------------
namespace {
// counter buffers of a region, taken in turn by the steps: with three of them the genotype kernel of step k (which
// waits for every rank's filter k) can run beside the filter of step k + 1 on another stream
constexpr uint32_t XCHG_BUFS = 3;
size_t xchg_counts_bytes(uint32_t num_sv) { return (size_t(num_sv) * 8 + 255) & ~size_t(255); }

__global__ void xchg_signal_kernel(Xchg x) {
    // the counters were written by kernels in front of this one on the same stream
    __threadfence_system();
    if (threadIdx.x < x.world) x.flags[threadIdx.x][x.rank] = x.epoch;
}
}  // namespace

extern "C" int svjg_xchg_create(uint32_t num_sv, void **d_base, uint8_t *ipc_handle64) {
    if (!d_base || !ipc_handle64) return svjg::set_error(SVJG_E_ARG, "svjg_xchg_create: NULL argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle is 64 bytes");
    const size_t bytes = XCHG_FLAG_WORDS * 4 + XCHG_BUFS * xchg_counts_bytes(num_sv);
    void *p = nullptr;
    SVJG_CUDA(cudaMalloc(&p, bytes));
    SVJG_CUDA(cudaMemset(p, 0, bytes));
    cudaIpcMemHandle_t h;
    SVJG_CUDA(cudaIpcGetMemHandle(&h, p));
    memcpy(ipc_handle64, &h, 64);
    *d_base = p;
    return SVJG_OK;
}
extern "C" int svjg_xchg_open(const uint8_t *ipc_handle64, void **d_peer) {
    if (!d_peer || !ipc_handle64) return svjg::set_error(SVJG_E_ARG, "svjg_xchg_open: NULL argument");
    cudaIpcMemHandle_t h;
    memcpy(&h, ipc_handle64, 64);
    SVJG_CUDA(cudaIpcOpenMemHandle(d_peer, h, cudaIpcMemLazyEnablePeerAccess));
    return SVJG_OK;
}
extern "C" int svjg_xchg_close(void *d_peer) {
    if (d_peer) SVJG_CUDA(cudaIpcCloseMemHandle(d_peer));
    return SVJG_OK;
}
extern "C" int svjg_xchg_free(void *d_base) {
    if (d_base) SVJG_CUDA(cudaFree(d_base));
    return SVJG_OK;
}
extern "C" uint32_t *svjg_xchg_counts(void *d_base, uint32_t num_sv, uint32_t parity) {
    return reinterpret_cast<uint32_t *>(static_cast<uint8_t *>(d_base) + XCHG_FLAG_WORDS * 4 + (parity % XCHG_BUFS) * xchg_counts_bytes(num_sv));
}
extern "C" int svjg_xchg_signal(void *const *d_regions, uint32_t world, uint32_t rank, uint32_t epoch, void *stream) {
    if (!d_regions || world == 0 || world > XCHG_MAX || rank >= world) return svjg::set_error(SVJG_E_ARG, "svjg_xchg_signal: bad argument");
    Xchg x{};
    x.world = world;
    x.rank = rank;
    x.epoch = epoch;
    for (uint32_t q = 0; q < world; ++q) x.flags[q] = static_cast<volatile uint32_t *>(d_regions[q]);   // flag words come first
    xchg_signal_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(x);
    SVJG_CUDA(cudaGetLastError());
    return SVJG_OK;
}
extern "C" int svjg_genotype_xchg(void *const *d_regions, uint32_t world, uint32_t rank, uint32_t num_sv, uint32_t parity,
                                  uint32_t epoch, int signal, const uint32_t *d_sv_index, const uint8_t *d_svtype, uint32_t n,
                                  int64_t min_support, double log10_1me, double log10_e, double log10_half,
                                  const double *d_lut, uint32_t lut_nmax, const double *d_k_override, int64_t *d_pl,
                                  uint8_t *d_gt, uint32_t *d_ad2, uint8_t *d_flags, void *stream) {
    if (!d_regions || world == 0 || world > XCHG_MAX || rank >= world) return svjg::set_error(SVJG_E_ARG, "svjg_genotype_xchg: bad argument");
    if (!d_sv_index || !d_svtype || !d_lut || !d_pl || !d_gt || !d_ad2 || !d_flags)
        return svjg::set_error(SVJG_E_ARG, "svjg_genotype_xchg: NULL argument");
    Xchg x{};
    x.world = world;
    x.rank = rank;
    x.epoch = epoch;
    x.signal = signal ? 1u : 0u;
    for (uint32_t q = 0; q < world; ++q) {
        x.counts[q] = svjg_xchg_counts(d_regions[q], num_sv, parity);
        x.flags[q] = static_cast<volatile uint32_t *>(d_regions[q]);
    }
    int threads = 128;
    int blocks = int((uint64_t(n ? n : 1) + threads - 1) / threads);
    genotype_kernel<true><<<blocks, threads, 0, (cudaStream_t)stream>>>(nullptr, x, d_sv_index, d_svtype, n, min_support, log10_1me,
                                                                        log10_e, log10_half, d_lut, lut_nmax, d_k_override,
                                                                        d_pl, d_gt, d_ad2, d_flags);
    SVJG_CUDA(cudaGetLastError());
    return SVJG_OK;
}
extern "C" int svjg_xchg_timed_out(void *d_base, uint32_t *out) {
    if (!d_base || !out) return svjg::set_error(SVJG_E_ARG, "svjg_xchg_timed_out: NULL argument");
    uint32_t v = 0;
    SVJG_CUDA(cudaMemcpy(&v, static_cast<uint8_t *>(d_base) + (XCHG_FLAG_WORDS - 1) * 4, 4, cudaMemcpyDeviceToHost));
    *out = v == 0xDEADu;
    return SVJG_OK;
}
