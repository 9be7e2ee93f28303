// br_fft.cuh -- the CMux step on the FP64 pipe: an exact external product through a float64 FFT with the key split
// into two 16-bit limbs (DESIGN.md section 4, "FFT throughput kernel"; error bound in section 8).
//
// Why it is exact.  The step needs, for each output polynomial mo, the integer negacyclic convolution
//     c_mo = sum_{mi, j} d_{mi,j} * k_{mi,j,mo}   (mod X^1024 + 1),  reduced mod 2^32,
// with signed digits |d| <= 512 and Torus32 key coefficients k.  Split k = k_lo + 2^16 k_hi, |k_lo|, |k_hi| <= 2^15:
// each limb convolution is an integer below 4 * 1024 * 2^9 * 2^15 = 2^36 in magnitude, which a float64 FFT computes
// with an error far below 1/2 (DESIGN.md section 8), so rounding recovers it exactly, and
//     c_mo mod 2^32 = lo32(c_lo) + (lo32(c_hi) << 16).
// Rounding is one DADD of 1.5 * 2^52: the low 32 mantissa bits of the sum are round(x) mod 2^32.
//
// Negacyclic convolution through a 512-point complex FFT: a real polynomial a of degree < 1024 is folded and twisted,
//     z_j = (a_j + i a_{j+512}) * omega^j,  omega = exp(i pi / 1024),  j < 512,
// and Z = DFT_512(z) (kernel exp(+2 pi i jk / 512)) holds a(omega^(4k+1)), evaluations at half of the roots of
// X^1024 + 1 (the other half are their conjugates).  Products of evaluations are evaluations of the product mod
// X^1024 + 1; the inverse runs the conjugate DFT, which returns 512 z: the factor 1/512 lives in the key spectra.
//
// The 512-point DFT is 8 x 8 x 8, j = 64 j0 + 8 j1 + j2, k = k0 + 8 k1 + 64 k2:
//     pass 1 (task t = 8 j1 + j2):  DFT8 over j0 -> k0, times W^(t k0)              (W = exp(2 pi i / 512) = omega^4)
//     pass 2 (task t = 8 k0 + j2):  DFT8 over j1 -> k1, times W^(8 j2 k1)
//     pass 3 (task t = 8 k0 + k1):  DFT8 over j2 -> k2
// every pass in place: element (a, b, c) lives at index 64 a + 8 b + c, so the spectrum X[k0 + 8 k1 + 64 k2] ends at
// index 64 k0 + 8 k1 + k2.  The MAC is point-wise, so it never needs natural order; the key spectra are stored in the
// same order.  The inverse runs the mirror image (passes 3, 2, 1, each the conjugate DFT8 after the conjugate twiddle)
// and ends in natural order.  Index i is stored at i + i / 8: every warp access of the three passes is bank-conflict
// free.
//
// Pass 1 merges the twist into its twiddle.  With twist omega^(64 j0 + t) = omega^t e^(i pi j0 / 16),
//     W^(t k0) DFT8_k0(a'_(64 j0 + t) omega^(64 j0 + t)) = omega^(t (1 + 4 k0)) DFT8_k0(a'_(64 j0 + t) e^(i pi j0 / 16)),
// so a task multiplies its inputs by 8 compile-time constants e^(i pi j0 / 16) (j0 = 0 is free, j0 = 4 is a rot8) and
// its outputs by 8 entries of one per-thread table, tw[64 k0 + t] = omega^(t (1 + 4 k0)), which it loads once for both
// of its polynomials.  The inverse pass 1 does the conjugate: the conjugate twiddle that pass 2 of the inverse would
// apply to its outputs (same element, same thread) and the untwist's omega^(-t) are conj(tw) on its inputs, the
// conjugate constants on its outputs.
//
// Every function is __host__ __device__ and every floating-point operation is explicit (fma() where fused, __dadd_rn /
// __dmul_rn on the device, which nvcc never contracts; the host emulator is built with -ffp-contract=off), so the host
// emulation computes the same bits as the GPU.
#pragma once
#include "br_phases.cuh"
#include <math.h>
#include <string.h>

namespace nb {

constexpr int FFT_M = 512;                          // complex points per polynomial
constexpr int FFT_STRIDE = FFT_M + FFT_M / 8;       // complex slots per polynomial in shared memory (padding)
constexpr int FFT_KEY_SPECTRA = 16;                 // per key row: 8 planes m = (mi * 2 + j) * 2 + mo, x 2 limbs
constexpr int FFT_ROW_U64 = FFT_KEY_SPECTRA * FFT_M * 2;     // 16384 u64 = 128 KB per key row
constexpr double FFT_ROUND_MAGIC = 6755399441055744.0;      // 1.5 * 2^52
constexpr double FFT_DIGIT_BIAS = 4503599627370496.0 + 512.0; // 2^52 + 512
constexpr double FFT_SQRT1_2 = 0.70710678118654752440;
// cos(pi j0 / 16), 0 <= j0 <= 8 (sin(pi j0 / 16) = cos(pi (8 - j0) / 16)), each rounded once: the factors
// e^(i pi j0 / 16) of pass 1 (j0 = 0 and 4 are not multiplied by: identity and rot8)
NB_HDC double fft_cos16(int j)
{
    return j == 0 ? 1.0 : j == 1 ? 0.9807852804032304491262 : j == 2 ? 0.9238795325112867561282
         : j == 3 ? 0.8314696123025452370788 : j == 4 ? 0.7071067811865475244008 : j == 5 ? 0.5555702330196022247428
         : j == 6 ? 0.3826834323650897717285 : j == 7 ? 0.1950903220161282678483 : 0.0;
}

NB_HD int fft_pos(int i) { return i + (i >> 3); }

struct cplx { double re, im; };

NB_HD double d_add(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
NB_HD double d_sub(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}
NB_HD double d_mul(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
NB_HD double d_fma(double a, double b, double c) { return fma(a, b, c); }
NB_HD cplx c_add(cplx a, cplx b) { return {d_add(a.re, b.re), d_add(a.im, b.im)}; }
NB_HD cplx c_sub(cplx a, cplx b) { return {d_sub(a.re, b.re), d_sub(a.im, b.im)}; }
NB_HD cplx c_mul(cplx a, cplx w) { return {d_fma(a.re, w.re, -d_mul(a.im, w.im)), d_fma(a.re, w.im, d_mul(a.im, w.re))}; }
NB_HD cplx c_conj(cplx a) { return {a.re, -a.im}; }
// acc + a * b
NB_HD cplx c_mac(cplx acc, cplx a, cplx b)
{
    return {d_fma(a.re, b.re, d_fma(-a.im, b.im, acc.re)), d_fma(a.re, b.im, d_fma(a.im, b.re, acc.im))};
}

// u in [0, 2^32) -> the double 2^52 + u, without a conversion instruction
NB_HD double d_from_u32_biased(u32 u)
{
#if defined(__CUDA_ARCH__)
    return __hiloint2double(0x43300000, (int)u);
#else
    const unsigned long long b = 0x4330000000000000ull | u;
    double d;
    memcpy(&d, &b, 8);
    return d;
#endif
}
// round(x) mod 2^32 for |x| < 2^51
NB_HD u32 d_round_lo32(double x)
{
    const double r = d_add(x, FFT_ROUND_MAGIC);
#if defined(__CUDA_ARCH__)
    return (u32)__double2loint(r);
#else
    unsigned long long b;
    memcpy(&b, &r, 8);
    return (u32)b;
#endif
}

NB_HD cplx ld_c(const cplx *p)
{
#if defined(__CUDA_ARCH__)
    const double2 t = *reinterpret_cast<const double2 *>(p);
    return {t.x, t.y};
#else
    return *p;
#endif
}
NB_HD void st_c(cplx *p, cplx v)
{
#if defined(__CUDA_ARCH__)
    *reinterpret_cast<double2 *>(p) = make_double2(v.re, v.im);
#else
    *p = v;
#endif
}
NB_HD cplx ld_c_global(const cplx *p)
{
#if defined(__CUDA_ARCH__)
    const double2 t = __ldg(reinterpret_cast<const double2 *>(p));
    return {t.x, t.y};
#else
    return *p;
#endif
}

// by e^(s i pi / 4) = (1 + s i) / sqrt 2, s = +1 (INV = false) or -1
template <bool INV> NB_HD cplx c_rot8(cplx a)
{
    return INV ? cplx{d_mul(d_add(a.re, a.im), FFT_SQRT1_2), d_mul(d_sub(a.im, a.re), FFT_SQRT1_2)}
               : cplx{d_mul(d_sub(a.re, a.im), FFT_SQRT1_2), d_mul(d_add(a.re, a.im), FFT_SQRT1_2)};
}
// by e^(s i pi j0 / 16), 0 < j0 < 8 (a compile-time constant wherever the caller's loop is unrolled)
template <bool INV> NB_HD cplx c_rot16(cplx a, int j0)
{
    if (j0 == 4) return c_rot8<INV>(a);
    return c_mul(a, cplx{fft_cos16(j0), INV ? -fft_cos16(8 - j0) : fft_cos16(8 - j0)});
}

// 8-point DFT in place, natural order in and out: y_k = sum_j x_j e^(s 2 pi i jk / 8), s = +1 (INV = false) or -1.
// Radix 2, decimation in frequency; the only non-trivial constants are e^(+-i pi / 4) = (1 +- i) / sqrt 2.
template <bool INV> NB_HD void dft8(cplx *x)
{
    // by e^(s i pi / 2): s = +1: (a + ib) i = -b + ia; s = -1: b - ia
    auto rot4 = [](cplx a) -> cplx { return INV ? cplx{a.im, -a.re} : cplx{-a.im, a.re}; };
    auto rot8 = [](cplx a) -> cplx { return c_rot8<INV>(a); };
    cplx a[4], b[4];
    for (int j = 0; j < 4; j++) { a[j] = c_add(x[j], x[j + 4]); b[j] = c_sub(x[j], x[j + 4]); }
    b[1] = rot8(b[1]); b[2] = rot4(b[2]); b[3] = rot4(rot8(b[3]));
    // two 4-point DFTs (root e^(s i pi / 2)): outputs 2k from a, 2k + 1 from b
    cplx a0 = c_add(a[0], a[2]), a1 = c_add(a[1], a[3]), a2 = c_sub(a[0], a[2]), a3 = rot4(c_sub(a[1], a[3]));
    cplx b0 = c_add(b[0], b[2]), b1 = c_add(b[1], b[3]), b2 = c_sub(b[0], b[2]), b3 = rot4(c_sub(b[1], b[3]));
    x[0] = c_add(a0, a1); x[4] = c_sub(a0, a1); x[2] = c_add(a2, a3); x[6] = c_sub(a2, a3);
    x[1] = c_add(b0, b1); x[5] = c_sub(b0, b1); x[3] = c_add(b2, b3); x[7] = c_sub(b2, b3);
}

// ---- tables (host-computed once, read by host emulator and kernels alike) ----------------------------------------
// tw[k0 * 64 + t] = omega^(t (1 + 4 k0)) (pass 1, twist merged in), tw2[a * 8 + b] = W^(8 a b) (pass 2, symmetric);
// omega = e^(i pi / 1024), W = omega^4.  Laid out so that the 32 lanes of a warp read consecutive or identical entries.
struct FftTables {
    cplx tw[FFT_M];
    cplx tw2[64];
};

// the 8 pass-1 factors of task t, tw[k0] = omega^(t (1 + 4 k0))
NB_HD void fft_load_tw1(int t, const FftTables &T, cplx *tw)
{
    for (int k0 = 0; k0 < 8; k0++) tw[k0] = ld_c(&T.tw[64 * k0 + t]);
}

// ---- passes over one polynomial `f` (FFT_STRIDE complex slots) ----------------------------------------------------
// forward pass 1 from values already in registers: x[j0] = a'[64 j0 + t], the folded input before the twist
// (z[64 j0 + t] = x[j0] omega^(64 j0 + t)); tw from fft_load_tw1
NB_HD void fft_fwd1_store(int t, cplx *x, cplx *f, const cplx *tw)
{
    for (int j0 = 1; j0 < 8; j0++) x[j0] = c_rot16<false>(x[j0], j0);
    dft8<false>(x);
    for (int k0 = 0; k0 < 8; k0++) st_c(f + fft_pos(64 * k0 + t), c_mul(x[k0], tw[k0]));
}
NB_HD void fft_fwd2(int t, cplx *f, const FftTables &T)
{
    const int base = 64 * (t >> 3) + (t & 7), j2 = t & 7;
    cplx x[8];
    for (int j1 = 0; j1 < 8; j1++) x[j1] = ld_c(f + fft_pos(base + 8 * j1));
    dft8<false>(x);
    st_c(f + fft_pos(base), x[0]);
    for (int k1 = 1; k1 < 8; k1++) st_c(f + fft_pos(base + 8 * k1), c_mul(x[k1], T.tw2[k1 * 8 + j2]));
}
NB_HD void fft_fwd3(int t, cplx *f)
{
    cplx *g = f + fft_pos(8 * t);                       // 8 consecutive slots
    cplx x[8];
    for (int j2 = 0; j2 < 8; j2++) x[j2] = ld_c(g + j2);
    dft8<false>(x);
    for (int k2 = 0; k2 < 8; k2++) st_c(g + k2, x[k2]);
}
NB_HD void fft_inv3(int t, cplx *f, const FftTables &T)
{
    cplx *g = f + fft_pos(8 * t);
    const int k1 = t & 7;
    cplx x[8];
    for (int k2 = 0; k2 < 8; k2++) x[k2] = ld_c(g + k2);
    dft8<true>(x);
    st_c(g, x[0]);
    for (int j2 = 1; j2 < 8; j2++) st_c(g + j2, c_mul(x[j2], c_conj(T.tw2[j2 * 8 + k1])));
}
// (its output twiddle conj(W^(t' k0)), t' = 8 j1 + j2, is applied by fft_inv1_load)
NB_HD void fft_inv2(int t, cplx *f)
{
    const int base = 64 * (t >> 3) + (t & 7);
    cplx x[8];
    for (int k1 = 0; k1 < 8; k1++) x[k1] = ld_c(f + fft_pos(base + 8 * k1));
    dft8<true>(x);
    for (int j1 = 0; j1 < 8; j1++) st_c(f + fft_pos(base + 8 * j1), x[j1]);
}
// inverse pass 1 into registers, untwisted: x[j0] = 512 a'[64 j0 + t] (the 1/512 is in the key spectra); tw from
// fft_load_tw1.  conj(tw[k0]) = conj(W^(t k0)) omega^(-t): pass 2's twiddle and the untwist's omega^(-t).
NB_HD void fft_inv1_load(int t, const cplx *f, const cplx *tw, cplx *x)
{
    for (int k0 = 0; k0 < 8; k0++) x[k0] = c_mul(ld_c(f + fft_pos(64 * k0 + t)), c_conj(tw[k0]));
    dft8<true>(x);
    for (int j0 = 1; j0 < 8; j0++) x[j0] = c_rot16<true>(x[j0], j0);
}

// ---- the CMux step ------------------------------------------------------------------------------------------------
// Work area of one ciphertext: 4 spectra of FFT_STRIDE complex.  Before the MAC, slot q = mi * 2 + j holds the
// spectrum of digit polynomial j of ACC[mi]; after it, slot mo * 2 + limb holds output polynomial mo, key limb `limb`.

// forward pass 1 for both digit polynomials of ACC[mi]: task t < 64.  Rotation (X^a - 1) ACC, the unsigned digit
// u = d + 512 (decomp_udigit), u -> d as 2^52 + u - (2^52 + 512), fold, pass 1 with the twist merged in.
template <bool ROTATE>
NB_HD void fft_step_fwd1(int t, const i32 *acc, cplx *f2 /* the 2 digit slots of ACC[mi] */, const FftTables &T, int a)
{
    const int ar = a & (NTT_N - 1);
    const bool flip = (a >> 10) & 1;
    u32 tv[16];                                         // coefficient + decomposition offset, [j0] and [8 + j0] (+512)
    for (int h = 0; h < 16; h++) {
        const int idx = 64 * (h & 7) + t + 512 * (h >> 3);
        const i32 c = ROTATE ? rotate_minus_one(acc, idx, ar, flip) : acc[idx];
        tv[h] = (u32)c + (0x80000000u + (1u << 21));
    }
    cplx tw[8];
    fft_load_tw1(t, T, tw);
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int j = 0; j < 2; j++) {
        const int sh = 22 - 10 * j;
        cplx x[8];
        for (int j0 = 0; j0 < 8; j0++) {
            const double lo = d_sub(d_from_u32_biased((tv[j0] >> sh) & 1023u), FFT_DIGIT_BIAS);
            const double hi = d_sub(d_from_u32_biased((tv[8 + j0] >> sh) & 1023u), FFT_DIGIT_BIAS);
            x[j0] = cplx{lo, hi};
        }
        fft_fwd1_store(t, x, f2 + j * FFT_STRIDE, tw);
    }
}

// MAC at point i (stored index) for `ct` ciphertexts whose work areas are `stride` complex apart: 16 key spectra of the
// row, loaded once for all of them.  key: [m = (mi * 2 + j) * 2 + mo][limb][i], complex.
NB_HD void fft_step_mac(int i, cplx *w, int stride, int ct, const cplx *key)
{
    cplx k[16];
    for (int s = 0; s < 16; s++) k[s] = ld_c_global(key + s * FFT_M + i);
    const int pos = fft_pos(i);
    for (int c = 0; c < ct; c++) {
        cplx *f = w + c * stride + pos;
        cplx d[4];
        for (int q = 0; q < 4; q++) d[q] = ld_c(f + q * FFT_STRIDE);
        for (int o = 0; o < 4; o++) {                    // o = mo * 2 + limb; key index (q * 2 + mo) * 2 + limb
            const int mo = o >> 1, limb = o & 1;
            cplx acc = {0.0, 0.0};
            for (int q = 0; q < 4; q++) acc = c_mac(acc, d[q], k[(q * 2 + mo) * 2 + limb]);
            st_c(f + o * FFT_STRIDE, acc);
        }
    }
}

// Inverse pass 1 for both limbs of output polynomial mo (task t < 64) with the untwist, round, recombine, ACC += (or =).
// Reports the largest |x - round(x)| through *err_max when it is not null (host emulation only).
template <bool ACCUMULATE>
NB_HD void fft_step_inv1(int t, i32 *acc, const cplx *f2 /* slots (mo, limb 0), (mo, limb 1) */, const FftTables &T,
                         double *err_max = nullptr)
{
    u32 r[16];                                          // lo32(c_lo) + (lo32(c_hi) << 16), [j0] and [8 + j0] (+512)
    for (int h = 0; h < 16; h++) r[h] = 0;
    cplx tw[8];
    fft_load_tw1(t, T, tw);
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int limb = 0; limb < 2; limb++) {
        cplx x[8];
        fft_inv1_load(t, f2 + limb * FFT_STRIDE, tw, x);
        const int sh = 16 * limb;
        for (int j0 = 0; j0 < 8; j0++) {
            const cplx y = x[j0];
            r[j0] += d_round_lo32(y.re) << sh;
            r[8 + j0] += d_round_lo32(y.im) << sh;
#if !defined(__CUDA_ARCH__)
            if (err_max) {
                const double e0 = fabs(y.re - nearbyint(y.re)), e1 = fabs(y.im - nearbyint(y.im));
                if (e0 > *err_max) *err_max = e0;
                if (e1 > *err_max) *err_max = e1;
            }
#endif
        }
    }
    for (int h = 0; h < 16; h++) {
        const int idx = 64 * (h & 7) + t + 512 * (h >> 3);
        const u32 v = r[h];
        acc[idx] = ACCUMULATE ? (i32)((u32)acc[idx] + v) : (i32)v;
    }
}

// ---- key spectra ---------------------------------------------------------------------------------------------------
// one key polynomial k (1024 int32, natural order) -> its two limb spectra, scaled by 1/512 (exact), into
// out[limb * FFT_M + i] (stored index order).  `f` is a scratch polynomial of FFT_STRIDE slots; the three passes are
// separated by barriers on the device (the caller's loop on the host), so this is split into the three phases.
NB_HD void fft_key_phase1(int t, const i32 *k, int limb, cplx *f, const FftTables &T)
{
    cplx x[8];
    for (int j0 = 0; j0 < 8; j0++) {
        const int idx = 64 * j0 + t;
        double v[2];
        for (int h = 0; h < 2; h++) {
            const i32 c = k[idx + 512 * h];
            const i32 lo = (i32)(int16_t)(u32)c;                // [-2^15, 2^15)
            const i32 hi = (i32)(((long long)c - lo) >> 16);     // [-2^15, 2^15]
            v[h] = (double)(limb ? hi : lo);
        }
        x[j0] = cplx{v[0], v[1]};
    }
    cplx tw[8];
    fft_load_tw1(t, T, tw);
    fft_fwd1_store(t, x, f, tw);
}
NB_HD void fft_key_phase3_store(int t, cplx *f, cplx *out)
{
    fft_fwd3(t, f);
    for (int k2 = 0; k2 < 8; k2++) {
        const cplx v = ld_c(f + fft_pos(8 * t + k2));
        out[8 * t + k2] = cplx{d_mul(v.re, 1.0 / 512), d_mul(v.im, 1.0 / 512)};
    }
}

}  // namespace nb
