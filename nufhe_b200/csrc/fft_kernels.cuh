// fft_kernels.cuh -- the throughput shape of the fused bootstrap on the FP64 pipe (br_fft.cuh), and the key spectra it
// reads.  The kernel keeps everything of blind_rotate_kernel (kernels.cuh) but the CMux step: the gate prologue and the
// mod-switch in its head, sample extraction in its tail, the persistent ready-queue with chunked chains and the start-up
// stagger of single-wave launches.  The step is the FFT external product: the integer work left is rotation,
// decomposition, addressing and the ACC update, the transforms and the MAC run as DFMA / DADD / DMUL.
#pragma once
#include "kernels.cuh"
#include "br_fft.cuh"

namespace nb {

// CT ciphertexts per CTA on 128 x CT threads; they share every key-row read of the MAC
template <int CT_> struct BrFftCfg {
    static constexpr int CT = CT_, THREADS = 128 * CT_;
    static constexpr int CTAS_PER_SM = CT_ <= 2 ? 2 : 1;
};
#ifndef NB_FFT_CT
#define NB_FFT_CT 2
#endif
using BrFft = BrFftCfg<NB_FFT_CT>;

template <class Cfg> constexpr size_t br_fft_smem_bytes()
{
    return (size_t)Cfg::CT * 4 * FFT_STRIDE * sizeof(cplx) + sizeof(FftTables) + (size_t)Cfg::CT * 2 * NTT_N * sizeof(i32) + 64;
}

// Phase clocks (profiling builds only: -DNB_FFT_PHASE_CLOCKS, tools/fft_phases.py).  Thread 0 of each CTA sums the
// clock64() cycles it spends in each phase of the step (FFT_CLK_FWD1 .. FFT_CLK_INV1), waiting at the step's barriers
// (FFT_CLK_SYNC) and fetching the next rotation (FFT_CLK_OTHER), and counts the steps; at exit it adds them to
// g_fft_phase_clocks[blockIdx.x].  The shipped library has none of it: FftClocks is then empty.
enum { FFT_CLK_FWD1, FFT_CLK_FWD2, FFT_CLK_FWD3, FFT_CLK_MAC, FFT_CLK_INV3, FFT_CLK_INV2, FFT_CLK_INV1, FFT_CLK_SYNC,
       FFT_CLK_OTHER, FFT_CLK_STEPS, FFT_CLK_SLOTS };
#ifdef NB_FFT_PHASE_CLOCKS
constexpr int FFT_CLK_CTAS = 1024;
__device__ unsigned long long g_fft_phase_clocks[FFT_CLK_CTAS][FFT_CLK_SLOTS];
__shared__ unsigned long long s_fft_clk[FFT_CLK_SLOTS];     // thread 0's sums (shared memory: no registers held)
struct FftClocks {
    long long t = 0;
    NB_D void start() { t = clock64(); }
    NB_D void mark(int k) { const long long n = clock64(); if (threadIdx.x == 0) s_fft_clk[k] += n - t; t = n; }
    NB_D void flush(int tid)
    {
        if (tid == 0 && blockIdx.x < FFT_CLK_CTAS)
            for (int k = 0; k < FFT_CLK_SLOTS; k++) g_fft_phase_clocks[blockIdx.x][k] += s_fft_clk[k];
    }
};
#else
struct FftClocks {
    NB_D void start() {}
    NB_D void mark(int) {}
    NB_D void flush(int) {}
};
#endif

// one CMux step of the CTA's ciphertexts: ACC[ct] += key (x) ((X^rot[ct] - 1) ACC[ct]); key = the row's 16 spectra
template <class Cfg>
NB_D void br_fft_step(cplx *w, const FftTables &T, i32 *acc, const int *rot, const cplx *__restrict__ key, int tid, FftClocks &clk)
{
    constexpr int TH = Cfg::THREADS;
    {   // task (ct * 2 + mi, t): both digit polynomials of ACC[mi]
        const int pm = tid >> 6;
        fft_step_fwd1<true>(tid & 63, acc + pm * NTT_N, w + pm * 2 * FFT_STRIDE, T, rot[pm >> 1]);
    }
    clk.mark(FFT_CLK_FWD1);
    __syncthreads();
    clk.mark(FFT_CLK_SYNC);
#pragma unroll 1
    for (int it = 0; it < 2; it++) { const int task = it * TH + tid; fft_fwd2(task & 63, w + (task >> 6) * FFT_STRIDE, T); }
    clk.mark(FFT_CLK_FWD2);
    __syncthreads();
    clk.mark(FFT_CLK_SYNC);
#pragma unroll 1
    for (int it = 0; it < 2; it++) { const int task = it * TH + tid; fft_fwd3(task & 63, w + (task >> 6) * FFT_STRIDE); }
    clk.mark(FFT_CLK_FWD3);
    __syncthreads();
    clk.mark(FFT_CLK_SYNC);
#pragma unroll 1
    for (int i = tid; i < FFT_M; i += TH) fft_step_mac(i, w, 4 * FFT_STRIDE, Cfg::CT, key);
    clk.mark(FFT_CLK_MAC);
    __syncthreads();
    clk.mark(FFT_CLK_SYNC);
#pragma unroll 1
    for (int it = 0; it < 2; it++) { const int task = it * TH + tid; fft_inv3(task & 63, w + (task >> 6) * FFT_STRIDE, T); }
    clk.mark(FFT_CLK_INV3);
    __syncthreads();
    clk.mark(FFT_CLK_SYNC);
#pragma unroll 1
    for (int it = 0; it < 2; it++) { const int task = it * TH + tid; fft_inv2(task & 63, w + (task >> 6) * FFT_STRIDE); }
    clk.mark(FFT_CLK_INV2);
    __syncthreads();
    clk.mark(FFT_CLK_SYNC);
    {   // task (ct * 2 + mo, t): both limbs of output polynomial mo
        const int pp = tid >> 6;
        fft_step_inv1<true>(tid & 63, acc + pp * NTT_N, w + pp * 2 * FFT_STRIDE, T);
    }
    clk.mark(FFT_CLK_INV1);
}

// Gate bootstraps only (p.bara == null, p.plain == 0): the key handle holds the n NTT rows and, after them, the n rows of
// spectra (nb_bk_prepare), so p.n is also the row count.  Queue, chunks and stagger: see blind_rotate_kernel.
template <class Cfg>
__global__ void __launch_bounds__(Cfg::THREADS, Cfg::CTAS_PER_SM) blind_rotate_fft_kernel(BlindRotateArgs p, const FftTables *__restrict__ tab_g)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cplx *w = reinterpret_cast<cplx *>(smem_raw);
    FftTables &T = *reinterpret_cast<FftTables *>(w + Cfg::CT * 4 * FFT_STRIDE);
    i32 *acc = reinterpret_cast<i32 *>(&T + 1);
    int *rot = reinterpret_cast<int *>(acc + Cfg::CT * 2 * NTT_N);
    __shared__ unsigned s_item, s_entry;
    const int tid = threadIdx.x;
    FftClocks clk;
#ifdef NB_FFT_PHASE_CLOCKS
    if (tid < FFT_CLK_SLOTS) s_fft_clk[tid] = 0;
#endif
    for (int i = tid; i < (int)(sizeof(FftTables) / 16); i += Cfg::THREADS)
        reinterpret_cast<double2 *>(&T)[i] = reinterpret_cast<const double2 *>(tab_g)[i];
    const cplx *key0 = reinterpret_cast<const cplx *>(p.bk + (size_t)p.n * BK_ROW_U64);
    constexpr int KEY_ROW_CPLX = FFT_KEY_SPECTRA * FFT_M;
    const unsigned total = p.chains * p.chunks;
    constexpr int ACC_WORDS = Cfg::CT * 2 * NTT_N;
    if (Cfg::CTAS_PER_SM > 1 && !p.sched && p.stagger_cycles > 0 && blockIdx.x >= (unsigned)p.sm_count) {
        if (tid == 0) {
            const long long t0 = clock64();
            while (clock64() - t0 < p.stagger_cycles) { }
        }
    }
    __syncthreads();

    for (unsigned item = blockIdx.x;; ) {
        if (p.sched) {
            __syncthreads();
            if (tid == 0) s_item = atomicAdd(p.sched, 1u);
            __syncthreads();
            item = s_item;
        }
        if (item >= total) break;
        unsigned chunk = 0, chain = item;
        if (p.sched && item >= p.chains) {
            if (tid == 0) {
                unsigned e;
                while ((e = ld_acquire_u32(p.sched + BR_SCHED_HEADER + item)) == 0) __nanosleep(100);
                s_entry = e - 1;
            }
            __syncthreads();
            const unsigned e = s_entry;
            chunk = e / p.chains; chain = e - chunk * p.chains;
        }
        const size_t ct0 = (size_t)chain * Cfg::CT;
        auto ct_of = [&](int slot) { size_t c = ct0 + slot; return c < p.batch ? c : p.batch - 1; };
        const int step0 = (int)chunk * p.steps_per_chunk;
        const int step1 = min(p.n, step0 + p.steps_per_chunk);

        if (chunk == 0) {
            for (int e = tid; e < ACC_WORDS; e += Cfg::THREADS) {
                const int slot = e >> 11, mi = (e >> 10) & 1, x = e & (NTT_N - 1);
                acc[e] = br2_initial_acc(p, ct_of(slot), mi, x);
            }
        } else {
            const int4 *src = reinterpret_cast<const int4 *>(p.state + (size_t)chain * ACC_WORDS);
            for (int e = tid; e < ACC_WORDS / 4; e += Cfg::THREADS) reinterpret_cast<int4 *>(acc)[e] = __ldcg(src + e);
        }
        if (tid < Cfg::CT) rot[(step0 & 1) * Cfg::CT + tid] = br2_rotation(p, ct_of(tid), step0);
        __syncthreads();
        clk.start();
        for (int i = step0; i < step1; i++) {
            int next = 0;
            if (tid < Cfg::CT && i + 1 < step1) next = br2_rotation(p, ct_of(tid), i + 1);
            clk.mark(FFT_CLK_OTHER);
            br_fft_step<Cfg>(w, T, acc, rot + (i & 1) * Cfg::CT, key0 + (size_t)i * KEY_ROW_CPLX, tid, clk);
            if (tid < Cfg::CT) rot[((i + 1) & 1) * Cfg::CT + tid] = next;
            __syncthreads();
            clk.mark(FFT_CLK_SYNC);
        }
#ifdef NB_FFT_PHASE_CLOCKS
        if (tid == 0) s_fft_clk[FFT_CLK_STEPS] += step1 - step0;
#endif

        if (step1 < p.n) {
            int4 *dst = reinterpret_cast<int4 *>(p.state + (size_t)chain * ACC_WORDS);
            for (int e = tid; e < ACC_WORDS / 4; e += Cfg::THREADS) __stcg(dst + e, reinterpret_cast<const int4 *>(acc)[e]);
            __threadfence();
            __syncthreads();
            if (tid == 0) {
                const unsigned slot = p.chains + atomicAdd(p.sched + 1, 1u);
                st_release_u32(p.sched + BR_SCHED_HEADER + slot, 1u + chain + p.chains * (chunk + 1));
            }
        } else {
            for (int e = tid; e < ACC_WORDS; e += Cfg::THREADS) {
                const int slot = e >> 11, mi = (e >> 10) & 1, x = e & (NTT_N - 1);
                const size_t c = ct0 + slot;
                if (c >= p.batch) continue;
                if (p.accum_out) p.accum_out[(c * 2 + mi) * NTT_N + x] = acc[e];
                if (p.extract) {
                    const i32 *a0 = acc + slot * 2 * NTT_N;
                    if (mi == 0) p.out_a[c * NTT_N + x] = x == 0 ? a0[0] : (i32)(0u - (u32)a0[NTT_N - x]);
                    else if (x == 0) p.out_b[c] = a0[NTT_N];
                }
            }
        }
        if (!p.sched) break;
    }
    clk.flush(tid);
}

// ---- key spectra (nb_bk_prepare) ------------------------------------------------------------------------------------
// reference Montgomery NTT values -> plain values, natural order (the input of ntt_inverse_kernel<true>)
__global__ void bk_plain_kernel(const u64 *__restrict__ bk_ref, u64 *__restrict__ out, size_t n)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        out[i] = ff_mul(ff_canon(bk_ref[i]), FF_RINV);
}

// one CTA of 64 threads per (key polynomial, limb): k (int32 coefficients, natural order) -> limb spectrum / 512
__global__ void __launch_bounds__(64) fft_key_kernel(const i32 *__restrict__ k, cplx *__restrict__ out, const FftTables *__restrict__ tab_g)
{
    __shared__ __align__(16) cplx f[FFT_STRIDE];
    const size_t poly = blockIdx.x >> 1;
    const int limb = blockIdx.x & 1, t = threadIdx.x;
    const FftTables &T = *tab_g;
    fft_key_phase1(t, k + poly * NTT_N, limb, f, T);
    __syncthreads();
    fft_fwd2(t, f, T);
    __syncthreads();
    fft_key_phase3_store(t, f, out + (size_t)blockIdx.x * FFT_M);
}

}  // namespace nb
