/*
 * nufhe_b200.h -- C ABI of libnufhe_b200.so, the B200 (sm_100a) engine for the gate-bootstrapping hot
 * path of nucypher/nufhe.
 *
 * The reference has no FFI: its boundary is the set of Python call signatures listed in SURVEY.md
 * section 8(b).  Each entry point below replaces the device work behind one of them; the reference
 * file:line is cited next to it.  All array arguments are caller-owned, dense, C-contiguous DEVICE
 * pointers (torch `data_ptr()` / cudaMalloc) unless a name ends in `_host`; the library allocates only
 * inside nb_ctx (constant tables and per-call scratch).  Every call enqueues work on the context's
 * stream and returns without synchronising.  Return value: 0 on success, negative NB_E* otherwise;
 * nb_last_error() gives the message.  No torch types, no C++ types.
 *
 * Layouts (SURVEY.md Appendix C): LWE sample a:(B,n) int32, b:(B,) int32; TLWE accumulator (B,2,1024)
 * int32; reference bootstrap key (n,2,2,2,1024) uint64 = NTT(bk)*2^64 mod p in natural order; key-switch
 * key a:(1024,t,base,n) int32, b:(1024,t,base) int32, cv:(1024,t,base) float32.
 */
#ifndef NUFHE_B200_H
#define NUFHE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NB_OK 0
#define NB_EINVAL (-1)       /* bad argument (Python shim raises ValueError) */
#define NB_EUNSUPPORTED (-2) /* parameter set outside the built path (ValueError, as blind_rotate.py:37-86) */
#define NB_ECUDA (-3)        /* CUDA runtime error (RuntimeError) */

typedef struct nb_ctx nb_ctx;

/* Replaces the Reikna Thread of a nufhe.Context (api_high_level.py:153-181): binds (device, stream).
 * `stream` is a cudaStream_t (0 = default stream). */
int nb_ctx_create(int device, void *stream, nb_ctx **out);
void nb_ctx_destroy(nb_ctx *ctx);
const char *nb_last_error(const nb_ctx *ctx);
int nb_ctx_set_stream(nb_ctx *ctx, void *stream);
/* Pre-allocate the context's scratch (work queue and parked accumulators of the fused bootstrap, variance block sums
 * of the key switch) for launches of up to `batch` ciphertexts.  Calls within that size then allocate nothing, which
 * is what CUDA-graph capture of a gate circuit needs (reference counterpart: Reikna plans allocate their temporaries
 * when a computation is compiled, blind_rotate.py:245-246). */
int nb_ctx_reserve(nb_ctx *ctx, size_t batch);
int nb_ctx_synchronize(nb_ctx *ctx);          /* thread.synchronize() */
/* Library / device facts: sm count, kernel register counts etc. as a short text (for bench/profiles). */
const char *nb_build_info(void);

/* ---- transform: nufhe/transform/computation.py:28-99 `Transform` (natural order in and out) ---- */
/* ForwardTransform (polynomial_transform_ntt.py:120-124): int32 coefficients -> field, i32_conversion=True */
int nb_ntt_forward_i32(nb_ctx *ctx, const int32_t *in, uint64_t *out, size_t batch);
/* Transform(inverse=False, i32_conversion=False) */
int nb_ntt_forward_u64(nb_ctx *ctx, const uint64_t *in, uint64_t *out, size_t batch);
/* InverseTransform (polynomial_transform_ntt.py:127-131) */
int nb_ntt_inverse_i32(nb_ctx *ctx, const uint64_t *in, int32_t *out, size_t batch);
int nb_ntt_inverse_u64(nb_ctx *ctx, const uint64_t *in, uint64_t *out, size_t batch);

/* ---- field arithmetic: nufhe/transform/arithmetic.py:56-270 (element-wise; op codes below).
 * b may have b_period elements (broadcast, i % b_period) or be NULL for unary ops. */
#define NB_FF_ADD 0
#define NB_FF_SUB 1
#define NB_FF_MUL 2
#define NB_FF_MUL_PREPARED 3 /* a*b*2^-64, arithmetic.mako:355-419 */
#define NB_FF_PREPARE 4      /* a*2^64,    arithmetic.mako:336-352 */
#define NB_FF_LSH 5          /* a*2^b, b < 192, arithmetic.mako:465-1045 */
#define NB_FF_LSH_CONST 6    /* same result through the compile-time-shift code paths the transforms use */
int nb_ff_elementwise(nb_ctx *ctx, int op, const uint64_t *a, const uint64_t *b, uint64_t *out, size_t n,
                      size_t b_period);

/* ---- bootstrap key: BootstrapKey / TransformedTGswSampleArray (bootstrap.py:44-92, tgsw.py:99-130).
 * Re-lays `rows` reference rows (each 2*2*2*1024 uint64) into the engine's internal row format:
 * nb_bk_row_u64() uint64 per row: the NTT part (the 8 planes re-ordered and un-Montgomery-ed + 2 correction planes,
 * 10 x 1024) and the FFT part (the 16 float64 limb spectra of the row, 16384).  bk_int holds all `rows` NTT parts first,
 * then all FFT parts; the gate entry points with LWE dimension n read a key of exactly n rows. */
size_t nb_bk_row_u64(void);
int nb_bk_prepare(nb_ctx *ctx, const uint64_t *bk_ref, uint64_t *bk_int, size_t rows);

/* ---- tgsw_transformed_external_mul (tgsw.py:165-172): accum (B,2,1024) <- bk[row] (x) accum ---- */
int nb_external_product(nb_ctx *ctx, int32_t *accum, const uint64_t *bk_int, size_t bk_row, size_t batch);

/* ---- BlindRotate_gpu (blind_rotate.py:262-281) without the key switch: explicit accumulator and bara.
 * out_a (B,1024), out_b (B,) receive the extracted samples; accum_out (optional) the rotated accumulators. */
int nb_blind_rotate(nb_ctx *ctx, const int32_t *accum, const int32_t *bara, const uint64_t *bk_int, size_t n,
                    int32_t *out_a, int32_t *out_b, int32_t *accum_out, size_t batch);

/* ---- bootstrap (bootstrap.py:206-229) fused with the gates' linear prologue (gates.py:108-115 etc.):
 * x = (0, c) + s1 * in1 + s2 * in2  (in2 may be NULL), then mod-switch, test vector, blind rotation and
 * sample extraction in one kernel.  Output: extracted LWE sample a:(B,1024), b:(B,). */
int nb_bootstrap_extract(nb_ctx *ctx, const int32_t *in1_a, const int32_t *in1_b, const int32_t *in2_a,
                         const int32_t *in2_b, int32_t c, int32_t s1, int32_t s2, int32_t mu,
                         const uint64_t *bk_int, size_t n, int32_t *out_a, int32_t *out_b, size_t batch);

/* Two bootstraps in one launch (gate_mux, gates.py:638-655): job A on ciphertexts [0, B), job B on [B, 2B);
 * out_a (2B,1024), out_b (2B,).  Halves the latency of small-batch MUX gates. */
int nb_bootstrap_extract2(nb_ctx *ctx, const int32_t *a1_a, const int32_t *a1_b, const int32_t *a2_a,
                          const int32_t *a2_b, int32_t a_c, int32_t a_s1, int32_t a_s2, const int32_t *b1_a,
                          const int32_t *b1_b, const int32_t *b2_a, const int32_t *b2_b, int32_t b_c, int32_t b_s1,
                          int32_t b_s2, int32_t mu, const uint64_t *bk_int, size_t n, int32_t *out_a, int32_t *out_b,
                          size_t batch);

/* ---- lwe_keyswitch (lwe.py:311-322): res = keyswitch((0, c) + src1 + src2), src2 may be NULL.
 * res_cv may be NULL. */
int nb_keyswitch(nb_ctx *ctx, const int32_t *src1_a, const int32_t *src1_b, const int32_t *src2_a,
                 const int32_t *src2_b, int32_t c, const int32_t *ks_a, const int32_t *ks_b, const float *ks_cv,
                 size_t in_size, size_t n, int t, int log2_base, int32_t *res_a, int32_t *res_b, float *res_cv,
                 size_t batch);

/* ---- LweLinear / LweNoiselessTrivial (lwe.py:346-422): res = (0, c) + s1 * x1 + s2 * x2 ------- */
int nb_lwe_affine(nb_ctx *ctx, int32_t *res_a, int32_t *res_b, const int32_t *x1_a, const int32_t *x1_b,
                  const int32_t *x2_a, const int32_t *x2_b, int32_t c, int32_t s1, int32_t s2, size_t batch,
                  size_t n);

/* ---- the separate steps of the multi-kernel bootstrap (bootstrap.py:96-196), `single_kernel_bootstrap=False` ---- */
/* ShiftTorusPolynomial (polynomials.py:90-104, polynomials_gpu.mako:18-77).  mode NB_SHIFT_INVERT: result =
 * X^(2N - power) * source (shift_tp_inverted_power); NB_SHIFT_MINUS_ONE: (X^power - 1) * source
 * (shift_tp_minus_one_power_from_array / tlwe_shift_polynomials); NB_SHIFT_PLAIN: X^power * source.
 * source/result: (polys, N) int32, N = 2^n_log2.  Polynomial p uses
 * powers[(p / polys_per_power) * powers_stride + power_idx]. */
#define NB_SHIFT_INVERT 0
#define NB_SHIFT_MINUS_ONE 1
#define NB_SHIFT_PLAIN 2
int nb_shift_torus_polynomial(nb_ctx *ctx, int32_t *result, const int32_t *source, const int32_t *powers,
                              size_t powers_stride, size_t power_idx, int polys_per_power, int mode, int n_log2,
                              size_t polys);
/* tlwe_noiseless_trivial (tlwe.py:156-158): acc (B, k+1, N) = (0, .., 0, mu (B, N)); cv (B,) = 0, one variance per
 * sample (may be NULL) */
int nb_tlwe_noiseless_trivial(nb_ctx *ctx, int32_t *acc, float *cv, const int32_t *mu, int mask_size, int n_log2,
                              size_t batch);
/* tlwe_extract_lwe_samples (tlwe.py:161-165): out_a (B, k*N), out_b (B,) from acc (B, k+1, N) */
int nb_tlwe_extract_lwe_samples(nb_ctx *ctx, int32_t *out_a, int32_t *out_b, const int32_t *acc, int mask_size,
                                int n_log2, size_t batch);
/* t32_to_phase (numeric_functions.py:34-36, kernel numeric_functions_gpu.py:39-77): the mod-switch of bootstrap()
 * (bootstrap.py:216-219) as a separate step; mspace_size must divide 2^32 */
int nb_t32_to_phase(nb_ctx *ctx, int32_t *out, const int32_t *in, size_t n, uint32_t mspace_size);
/* The external product of the multi-kernel path step by step (TGswTransformedExternalMul, tgsw_gpu.py:110-169), for
 * any TLWE mask size k and decomposition length l -- the fused kernel covers k = 1, l = 2 only:
 * decompose -> nb_ntt_forward_i32 -> MAC -> nb_ntt_inverse_i32.
 * nb_tgsw_decompose (tgsw_gpu.py:31-54): out (polys, l, N) from in (polys, N); offset = TGswParams.offset.
 * nb_tgsw_mac (tgsw_gpu.py:58-107): out (B, k+1, 1024) = sum_{mi,j} mul_prepared(tr (B, k+1, l, 1024),
 * bk_row (k+1, l, k+1, 1024)), bk_row in the reference's layout (natural order, Montgomery form). */
int nb_tgsw_decompose(nb_ctx *ctx, int32_t *out, const int32_t *in, size_t polys, int decomp_length, int bs_log2_base,
                      int32_t offset, int n_log2);
int nb_tgsw_mac(nb_ctx *ctx, uint64_t *out, const uint64_t *tr, const uint64_t *bk_row, size_t batch, int mask_size,
                int decomp_length);
/* tlwe_add_to (tlwe.py:173-175): res += src (int32 wrap-around, n elements); variances (n_cv floats, may be NULL) */
int nb_tlwe_add_to(nb_ctx *ctx, int32_t *res, const int32_t *src, size_t n, float *res_cv, const float *src_cv,
                   size_t n_cv);

/* LweEncrypt / LweDecrypt (lwe_gpu.py:186-284, kernels lwe_gpu.mako:205-262; lwe.py:325-343): the wrap-around dot
 * product of LWE masks a (B, n) with the binary key (n),
 *     out[i] = add1[i] (+ add2[i]) + sign * <a[i, :], key>       (add1, add2 may be NULL)
 * encrypt: out = b, add1 = messages, add2 = noises_b, sign = +1;  decrypt phase: add1 = b, sign = -1. */
int nb_lwe_dot(nb_ctx *ctx, int32_t *out, const int32_t *a, const int32_t *key, const int32_t *add1,
               const int32_t *add2, int32_t sign, size_t batch, size_t n);
/* MakeLweKeyswitchKey (lwe_gpu.py:63-124, kernel lwe_gpu.mako:18-56; lwe.py:265-295): ks_a (in, t, base, n),
 * ks_b / ks_cv (in, t, base) from in_key (in), out_key (n), noises_a (in, t, base-1, n), noises_b (in, t, base-1):
 * row h = 0 is zero, row h encrypts in_key[i] * h * 2^(32 - (j+1) log2_base) with variance noise_variance. */
int nb_make_keyswitch_key(nb_ctx *ctx, int32_t *ks_a, int32_t *ks_b, float *ks_cv, const int32_t *in_key,
                          const int32_t *out_key, const int32_t *noises_a, const int32_t *noises_b, size_t in_size,
                          size_t n, int t, int log2_base, float noise_variance);

#ifdef __cplusplus
}
#endif
#endif
