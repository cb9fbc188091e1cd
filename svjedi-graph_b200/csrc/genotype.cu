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
__device__ __forceinline__ void genotype_one(uint32_t n0, uint32_t n1, uint32_t idx, uint32_t ty, int64_t min_support,
                                             double la, double lb, double lh, const double *lut, uint32_t lut_nmax,
                                             const double *k_override, size_t o, int64_t *pl, uint8_t *gt,
                                             uint32_t *ad2, uint8_t *flags) {
    // predict-genotype.py:216 — a key is "in the dict" once it has at least one hit
    bool gate = (ty & 0x3F) <= 3 && !(ty & 0x80) && ty != 255 && idx != 0xFFFFFFFFu && ((n0 | n1) != 0 || (ty & 0x40));
    if (!gate) {
        gt[o] = 3;
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
    genotype_one(n0, n1, idx, ty, min_support, la, lb, lh, lut, lut_nmax, k_override, i, pl, gt, ad2, flags);
}

// One thread per cell (record i, sample s) of a block of records.  The counters are the cohort's sample-major
// matrix ([S][num_sv][2], as the filter writes a sample's counters); the results are record-major ([n][S], the
// order of the VCF text).
__global__ void genotype_cohort_kernel(const uint32_t *__restrict__ counts, uint32_t num_sv, uint32_t n_samples,
                                       const uint32_t *__restrict__ sv_index, const uint8_t *__restrict__ svtype,
                                       uint32_t n_cells, int64_t min_support, double la, double lb, double lh,
                                       const double *__restrict__ lut, uint32_t lut_nmax, int64_t *__restrict__ pl,
                                       uint8_t *__restrict__ gt, uint32_t *__restrict__ ad2, uint8_t *__restrict__ flags) {
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
    genotype_one(n0, n1, idx, svtype[i], min_support, la, lb, lh, lut, lut_nmax, nullptr, c, pl, gt, ad2, flags);
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
// along the row, one warp reduction), then every thread runs the exact tests of one record, which are serial per
// record.  Results: gcount[i] = (r0, h, r2, missing), hwe[i], exchet[i].
constexpr int SITE_THREADS = 256;
__global__ void __launch_bounds__(SITE_THREADS)
cohort_site_stats_kernel(const uint8_t *__restrict__ gt, uint32_t n, uint32_t n_samples, uint4 *__restrict__ gcount,
                         double *__restrict__ hwe, double *__restrict__ exchet) {
    __shared__ uint32_t cnt[3][SITE_THREADS];
    const uint32_t base = blockIdx.x * SITE_THREADS, lane = threadIdx.x & 31;
    for (uint32_t r = threadIdx.x >> 5; r < SITE_THREADS && base + r < n; r += SITE_THREADS / 32) {
        const uint8_t *row = gt + size_t(base + r) * n_samples;
        uint32_t c0 = 0, c1 = 0, c2 = 0;
        for (uint32_t s = lane; s < n_samples; s += 32) {
            const uint32_t g = row[s];
            c0 += g == 0;
            c1 += g == 1;
            c2 += g == 2;
        }
        c0 = __reduce_add_sync(0xFFFFFFFFu, c0);
        c1 = __reduce_add_sync(0xFFFFFFFFu, c1);
        c2 = __reduce_add_sync(0xFFFFFFFFu, c2);
        if (lane == 0) {
            cnt[0][r] = c0;
            cnt[1][r] = c1;
            cnt[2][r] = c2;
        }
    }
    __syncthreads();
    const uint32_t i = base + threadIdx.x;
    if (i >= n) return;
    const uint32_t r0 = cnt[0][threadIdx.x], h = cnt[1][threadIdx.x], r2 = cnt[2][threadIdx.x];
    gcount[i] = make_uint4(r0, h, r2, n_samples - r0 - h - r2);
    double p_hwe, p_exc;
    site_exact_tests(r0, h, r2, p_hwe, p_exc);
    hwe[i] = p_hwe;
    exchet[i] = p_exc;
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
extern "C" int svjg_cohort_genotype(svjg_cohort *c, const uint32_t *sv_index, const uint8_t *svtype, uint32_t n,
                                    int64_t min_support, double log10_1me, double log10_e, double log10_half,
                                    const double *lut, uint32_t lut_nmax, int64_t *pl, uint8_t *gt, uint32_t *ad2,
                                    uint8_t *flags) {
    if (!c) return svjg::set_error(SVJG_E_ARG, "svjg_cohort_genotype: NULL cohort");
    c->blk_n = 0;                          // set again once this block's cells are complete
    if (n == 0) return SVJG_OK;
    if (!sv_index || !svtype || !lut || !pl || !gt || !ad2 || !flags)
        return svjg::set_error(SVJG_E_ARG, "svjg_cohort_genotype: NULL argument");
    if (!(log10_1me == log10_1me) || !(log10_e == log10_e) || !(log10_half == log10_half))
        return svjg::set_error(SVJG_E_ARG, "svjg_cohort_genotype: NaN constant");
    const uint64_t cells = uint64_t(n) * c->n_samples;
    if (cells >= 0xFFFFFFFFull) return svjg::set_error(SVJG_E_ARG, "svjg_cohort_genotype: block of more than 2^32 cells");
    for (uint32_t i = 0; i < n; ++i)
        if (sv_index[i] != 0xFFFFFFFFu && sv_index[i] >= c->num_sv)
            return svjg::set_error(SVJG_E_ARG, "svjg_cohort_genotype: sv_index out of range");
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
    const size_t b_idx = size_t(n) * 4, b_ty = n, b_pl = cells * 24, b_gt = cells, b_ad = cells * 8, b_fl = cells;
    const size_t o_ty = up(b_idx), o_pl = o_ty + up(b_ty), o_gt = o_pl + up(b_pl), o_ad = o_gt + up(b_gt),
                 o_fl = o_ad + up(b_ad), total = o_fl + up(b_fl);
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
    const int threads = 128;
    const uint32_t blocks = uint32_t((cells + threads - 1) / threads);
    genotype_cohort_kernel<<<blocks, threads, 0, st>>>(c->d_counts, c->num_sv, c->n_samples, reinterpret_cast<const uint32_t *>(d),
                                                       d + o_ty, uint32_t(cells), min_support, log10_1me, log10_e, log10_half,
                                                       c->d_lut, lut_nmax, reinterpret_cast<int64_t *>(d + o_pl), d + o_gt,
                                                       reinterpret_cast<uint32_t *>(d + o_ad), d + o_fl);
    SVJG_CUDA(cudaGetLastError());
    SVJG_CUDA(cudaMemcpyAsync(pl, d + o_pl, b_pl, cudaMemcpyDeviceToHost, st));
    SVJG_CUDA(cudaMemcpyAsync(gt, d + o_gt, b_gt, cudaMemcpyDeviceToHost, st));
    SVJG_CUDA(cudaMemcpyAsync(ad2, d + o_ad, b_ad, cudaMemcpyDeviceToHost, st));
    SVJG_CUDA(cudaMemcpyAsync(flags, d + o_fl, b_fl, cudaMemcpyDeviceToHost, st));
    SVJG_CUDA(cudaStreamSynchronize(st));
    c->blk_n = n;
    c->blk_gt = o_gt;
    return SVJG_OK;
}

// Site statistics of the block of the last svjg_cohort_genotype call, from its gt codes where the kernel left them
// on the device: 32 B per record come back, not the cells.
extern "C" int svjg_cohort_site_stats(svjg_cohort *c, uint32_t n, uint32_t *gcount, double *hwe, double *exchet) {
    if (!c) return svjg::set_error(SVJG_E_ARG, "svjg_cohort_site_stats: NULL cohort");
    if (n != c->blk_n)
        return svjg::set_error(SVJG_E_ARG, "svjg_cohort_site_stats: n is not the record count of the last svjg_cohort_genotype call");
    if (n == 0) return SVJG_OK;
    if (!gcount || !hwe || !exchet) return svjg::set_error(SVJG_E_ARG, "svjg_cohort_site_stats: NULL argument");
    // every D and E of the exact tests must be exact in a double
    const uint64_t s1 = uint64_t(c->n_samples) + 1;
    if (s1 >= (1ull << 26) || 4 * s1 * s1 >= (1ull << 53))
        return svjg::set_error(SVJG_E_ARG, "svjg_cohort_site_stats: 4 (S + 1)^2 must be below 2^53");
    SVJG_CUDA(cudaSetDevice(c->t->device));
    auto up = [](size_t x) { return (x + 255) & ~size_t(255); };
    const size_t b_cnt = size_t(n) * 16, b_p = size_t(n) * 8, o_hwe = up(b_cnt), o_exc = o_hwe + up(b_p), total = o_exc + up(b_p);
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
    cohort_site_stats_kernel<<<blocks, SITE_THREADS, 0, st>>>(c->d_blk + c->blk_gt, n, c->n_samples, reinterpret_cast<uint4 *>(d),
                                                              reinterpret_cast<double *>(d + o_hwe),
                                                              reinterpret_cast<double *>(d + o_exc));
    SVJG_CUDA(cudaGetLastError());
    SVJG_CUDA(cudaMemcpyAsync(gcount, d, b_cnt, cudaMemcpyDeviceToHost, st));
    SVJG_CUDA(cudaMemcpyAsync(hwe, d + o_hwe, b_p, cudaMemcpyDeviceToHost, st));
    SVJG_CUDA(cudaMemcpyAsync(exchet, d + o_exc, b_p, cudaMemcpyDeviceToHost, st));
    SVJG_CUDA(cudaStreamSynchronize(st));
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
