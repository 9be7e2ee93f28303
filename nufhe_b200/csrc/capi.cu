// capi.cu -- the C ABI of libnufhe_b200.so (see include/nufhe_b200.h).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <type_traits>
#include <nvtx3/nvToolsExt.h>
#include "../../include/nufhe_b200.h"
#include "kernels.cuh"
#include "fft_kernels.cuh"
#include "tables.h"

using namespace nb;

struct nb_ctx {
    int device;
    cudaStream_t stream;
    u64 *d_ph_fwd, *d_ph_inv;            // middle-twiddle tables [row][j2] of the transform passes
    u64 *d_ones512;                      // 512 * NTT(all-ones), natural order (bk_prepare)
    int sm_count;
    size_t wide_max;                     // largest batch launched in the wide (1 ciphertext / 256 threads) shape
    size_t wide2_max;                    // largest batch launched in the wide2 (1 ciphertext / 512 threads / SM) shape
    size_t pair_max;                     // largest batch launched in the pair shape (1 ciphertext / cluster of 2 CTAs on 2 SMs)
    int pair_async;                      // pair shape: exchange by st.async + mbarrier (1) or plain stores + barrier.cluster (0)
    int max_chunks;                      // upper bound on the chunks a chain is cut into (1 = no time slicing)
    unsigned *d_sched;                   // work-queue state of the fused bootstrap (kernels.cuh: BlindRotateArgs)
    size_t sched_words;
    int32_t *d_state;                    // parked accumulators of time-sliced launches
    size_t state_words;
    float *d_cv_blocks;                  // block sums of the key-switch variances (split launches)
    size_t cv_words;
    int force_chunks;                    // developer knob: chunk count of every multi-wave launch (0 = automatic)
    int stagger_cycles;                  // start-up offset of the second CTA per SM in single-wave launches
    int use_fft;                         // gate bootstraps above wide_max take the FP64 FFT kernel (fft_kernels.cuh)
    FftTables *d_fft_tab;                // its twiddle tables (br_fft.cuh)
    std::string err;
};

static int fail(nb_ctx *ctx, int code, const std::string &msg)
{
    if (ctx) ctx->err = msg;
    return code;
}

static int check(nb_ctx *ctx, cudaError_t e, const char *what)
{
    if (e == cudaSuccess) return NB_OK;
    return fail(ctx, NB_ECUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

#define NB_TRY(expr)                         \
    do {                                     \
        int _rc = (expr);                    \
        if (_rc != NB_OK) return _rc;        \
    } while (0)

static int launch_check(nb_ctx *ctx, const char *what) { return check(ctx, cudaGetLastError(), what); }

// Every entry point works on ctx->device and leaves the caller's current device as it found it (one process may
// hold several engines, one per GPU, like the reference's one-Context-per-device model, api_high_level.py:153-181).
struct DeviceGuard {
    int prev = -1;
    bool switched = false;
    cudaError_t err;
    explicit DeviceGuard(int dev)
    {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != dev) {
            err = cudaSetDevice(dev);
            switched = err == cudaSuccess;
        }
    }
    ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
};
// NVTX range around the launches of one entry point (prologue + blind rotation, key switch, transforms, ...): shows up
// in Nsight Systems / `ncu --nvtx`; a no-op costing two library calls when no tool is attached (nvtx3 is header-only).
struct NvtxRange {
    explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

#define NB_ON_DEVICE(ctx)                   \
    DeviceGuard _guard((ctx)->device);      \
    NB_TRY(check(ctx, _guard.err, "cudaSetDevice"))

extern "C" {

int nb_ctx_create(int device, void *stream, nb_ctx **out)
{
    if (!out) return NB_EINVAL;
    *out = nullptr;
    nb_ctx *ctx = new nb_ctx();
    ctx->device = device;
    ctx->stream = (cudaStream_t)stream;
    ctx->d_ph_fwd = ctx->d_ph_inv = ctx->d_ones512 = nullptr;
    ctx->d_sched = nullptr; ctx->d_state = nullptr; ctx->sched_words = ctx->state_words = 0;
    ctx->d_cv_blocks = nullptr; ctx->cv_words = 0;
    ctx->d_fft_tab = nullptr;
    *out = ctx;   // returned even on failure so that nb_last_error() can be read; caller destroys it
    NB_ON_DEVICE(ctx);
    cudaDeviceProp prop;
    NB_TRY(check(ctx, cudaGetDeviceProperties(&prop, device), "cudaGetDeviceProperties"));
    ctx->sm_count = prop.multiProcessorCount;
    {
        const char *e = getenv("NUFHE_B200_MAX_CHUNKS");  // developer knob: 1 disables the time slicing of chains
        ctx->max_chunks = e ? atoi(e) : 50;
        if (ctx->max_chunks < 1) ctx->max_chunks = 1;
        e = getenv("NUFHE_B200_FORCE_CHUNKS");
        ctx->force_chunks = e ? atoi(e) : 0;
        e = getenv("NUFHE_B200_STAGGER");
        ctx->stagger_cycles = e ? atoi(e) : 12000;        // about a quarter of a CMux step (measured best of 0 / 12k / 24k / 36k)
        e = getenv("NUFHE_B200_FFT");                      // 0: every batch stays on the NTT kernels
        ctx->use_fft = e ? atoi(e) : 1;
    }
    if (const char *e = getenv("NUFHE_B200_FORCE_RARE_PATH")) {
        // test knob: run the canonicalisation fix-up of the deferred-canonicalisation phases on every task
        if (atoi(e)) {
            const u32 zero = 0;
            NB_TRY(check(ctx, cudaMemcpyToSymbol(nb_c_canon_trigger, &zero, sizeof(zero)), "cudaMemcpyToSymbol"));
        }
    }
    if (prop.major < 10)
        return fail(ctx, NB_EUNSUPPORTED, "libnufhe_b200 is built for sm_100a only; device is sm_" +
                                              std::to_string(prop.major) + std::to_string(prop.minor));
    PhaseTables pt;
    NB_TRY(check(ctx, cudaMalloc(&ctx->d_ph_fwd, NTT_N * sizeof(u64)), "cudaMalloc"));
    NB_TRY(check(ctx, cudaMalloc(&ctx->d_ph_inv, NTT_N * sizeof(u64)), "cudaMalloc"));
    NB_TRY(check(ctx, cudaMemcpy(ctx->d_ph_fwd, pt.fwd.data(), NTT_N * sizeof(u64), cudaMemcpyHostToDevice), "memcpy"));
    NB_TRY(check(ctx, cudaMemcpy(ctx->d_ph_inv, pt.inv.data(), NTT_N * sizeof(u64), cudaMemcpyHostToDevice), "memcpy"));
    NB_TRY(check(ctx, cudaMalloc(&ctx->d_ones512, NTT_N * sizeof(u64)), "cudaMalloc"));
    NB_TRY(check(ctx, cudaMemcpy(ctx->d_ones512, pt.ones512.data(), NTT_N * sizeof(u64), cudaMemcpyHostToDevice), "memcpy"));
    {
        FftTables ft;
        make_fft_tables(ft);
        NB_TRY(check(ctx, cudaMalloc(&ctx->d_fft_tab, sizeof(FftTables)), "cudaMalloc"));
        NB_TRY(check(ctx, cudaMemcpy(ctx->d_fft_tab, &ft, sizeof(FftTables), cudaMemcpyHostToDevice), "memcpy"));
    }
    NB_TRY(check(ctx, cudaFuncSetAttribute(blind_rotate_fft_kernel<BrFft>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)br_fft_smem_bytes<BrFft>()), "cudaFuncSetAttribute(blind_rotate fft)"));
    NB_TRY(check(ctx, cudaFuncSetAttribute(blind_rotate_kernel<BrDefault>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)br_smem_bytes<BrDefault>()), "cudaFuncSetAttribute(blind_rotate)"));
    NB_TRY(check(ctx, cudaFuncSetAttribute(blind_rotate_kernel<BrWide>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)br_smem_bytes<BrWide>()), "cudaFuncSetAttribute(blind_rotate wide)"));
    NB_TRY(check(ctx, cudaFuncSetAttribute(blind_rotate_kernel<BrWide2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)br_smem_bytes<BrWide2>()), "cudaFuncSetAttribute(blind_rotate wide2)"));
    NB_TRY(check(ctx, cudaFuncSetAttribute(blind_rotate_pair_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)BR_PAIR_SMEM_BYTES), "cudaFuncSetAttribute(blind_rotate pair)"));
    NB_TRY(check(ctx, cudaFuncSetAttribute(blind_rotate_pair_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)BR_PAIR_SMEM_BYTES), "cudaFuncSetAttribute(blind_rotate pair)"));
    NB_TRY(check(ctx, cudaFuncSetAttribute(keyswitch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)KS_SMEM_BYTES), "cudaFuncSetAttribute(keyswitch)"));
    {   // batches that fit one wave of wide CTAs (one ciphertext on 256 threads) take the low-latency shape
        const char *e = getenv("NUFHE_B200_WIDE_MAX");
        // up to one wave the wide shape has the shortest step; between one and ~1.7 waves it still wins, time-sliced
        // over all SMs, against a throughput-shape launch that leaves half of the SMs with one CTA (r2 sweep)
        ctx->wide_max = e ? (size_t)atoll(e) : (size_t)ctx->sm_count * BrWide::CTAS_PER_SM * 17 / 10;
        // up to 1.5 ciphertexts per SM: 512 threads per ciphertext, forward phases split as well (lowest latency;
        // measured crossover against the 256-thread shape between 200 and 296 ciphertexts, profiles/r2_variants.md)
        e = getenv("NUFHE_B200_WIDE2_MAX");
        ctx->wide2_max = e ? (size_t)atoll(e) : (size_t)ctx->sm_count * 3 / 2;
        // up to one cluster of two SMs per ciphertext: the pair shape, while all clusters are resident at once (the
        // driver knows how many pairs of SMs it can form)
        e = getenv("NUFHE_B200_PAIR_ASYNC");
        ctx->pair_async = e ? atoi(e) : 1;
        e = getenv("NUFHE_B200_PAIR_MAX");
        if (e) {
            ctx->pair_max = (size_t)atoll(e);
        } else {
            cudaLaunchConfig_t cfg = {};
            cudaLaunchAttribute attr;
            attr.id = cudaLaunchAttributeClusterDimension;
            attr.val.clusterDim.x = 2; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
            cfg.gridDim = dim3(2 * (unsigned)ctx->sm_count); cfg.blockDim = dim3(PAIR_THREADS);
            cfg.dynamicSmemBytes = BR_PAIR_SMEM_BYTES; cfg.attrs = &attr; cfg.numAttrs = 1;
            int clusters = 0;
            if (cudaOccupancyMaxActiveClusters(&clusters, blind_rotate_pair_kernel<true>, &cfg) != cudaSuccess) {
                cudaGetLastError();
                clusters = 0;
            }
            // measured (profiles/r2_variants.md section 7): 3.0 ms against 4.0 ms up to 24 ciphertexts, 3.45 at 48, and
            // slower than the 512-thread shape at 64 (4.13 against 3.98) -- the more SMs of a GPC run, the less a shape
            // with 8 warps per SM hides; the crossover is near 3/8 ciphertexts per SM
            const size_t cap = (size_t)ctx->sm_count * 3 / 8;
            ctx->pair_max = clusters > 0 ? ((size_t)clusters < cap ? (size_t)clusters : cap) : 0;
        }
        if (getenv("NUFHE_B200_VERBOSE"))
            fprintf(stderr, "nufhe_b200: device %d, %d SMs; fused-kernel shapes by batch: pair <= %zu, wide2 <= %zu, wide <= %zu\n",
                    ctx->device, ctx->sm_count, ctx->pair_max, ctx->wide2_max, ctx->wide_max);
    }
    NB_TRY(check(ctx, cudaFuncSetAttribute(ntt_forward_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ntt_smem_bytes(NTT_RAW_I32_BYTES)), "attr"));
    NB_TRY(check(ctx, cudaFuncSetAttribute(ntt_forward_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ntt_smem_bytes(NTT_RAW_U64_BYTES)), "attr"));
    NB_TRY(check(ctx, cudaFuncSetAttribute(ntt_inverse_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ntt_smem_bytes(NTT_RAW_U64_BYTES)), "attr"));
    NB_TRY(check(ctx, cudaFuncSetAttribute(ntt_inverse_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ntt_smem_bytes(NTT_RAW_U64_BYTES)), "attr"));
    return NB_OK;
}

void nb_ctx_destroy(nb_ctx *ctx)
{
    if (!ctx) return;
    DeviceGuard guard(ctx->device);
    if (ctx->d_ph_fwd) cudaFree(ctx->d_ph_fwd);
    if (ctx->d_ph_inv) cudaFree(ctx->d_ph_inv);
    if (ctx->d_ones512) cudaFree(ctx->d_ones512);
    if (ctx->d_sched) cudaFree(ctx->d_sched);
    if (ctx->d_state) cudaFree(ctx->d_state);
    if (ctx->d_cv_blocks) cudaFree(ctx->d_cv_blocks);
    if (ctx->d_fft_tab) cudaFree(ctx->d_fft_tab);
    delete ctx;
}

const char *nb_last_error(const nb_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int nb_ctx_set_stream(nb_ctx *ctx, void *stream)
{
    if (!ctx) return NB_EINVAL;
    ctx->stream = (cudaStream_t)stream;
    return NB_OK;
}

int nb_ctx_synchronize(nb_ctx *ctx)
{
    if (!ctx) return NB_EINVAL;
    NB_ON_DEVICE(ctx);
    return check(ctx, cudaStreamSynchronize(ctx->stream), "cudaStreamSynchronize");
}

const char *nb_build_info(void)
{
    static std::string info;
    if (info.empty()) {
        char buf[512];
        cudaFuncAttributes a{}, b{}, c{};
        cudaFuncGetAttributes(&a, blind_rotate_kernel<BrDefault>);
        cudaFuncGetAttributes(&b, ntt_forward_kernel<true>);
        cudaFuncGetAttributes(&c, keyswitch_kernel);
        snprintf(buf, sizeof(buf),
                 "nufhe_b200 sm_100a; blind_rotate: %d regs, %zu B dyn smem, %d thr/CTA, %d ct/CTA; "
                 "ntt_forward: %d regs; keyswitch: %d regs, tile %d",
                 a.numRegs, BR2_SMEM_BYTES, BR2_THREADS, BR2_CT, b.numRegs, c.numRegs, KS_TILE);
        info = buf;
    }
    return info.c_str();
}

static int ntt_grid(nb_ctx *ctx, size_t batch)
{
    size_t blocks = (batch + NTT_SWEEP_POLYS - 1) / NTT_SWEEP_POLYS;
    size_t cap = (size_t)ctx->sm_count * NTT_CTAS;   // persistent: NTT_CTAS CTAs per SM, grid-stride over the batch
    return (int)(blocks < cap ? blocks : cap);
}

int nb_ntt_forward_i32(nb_ctx *ctx, const int32_t *in, uint64_t *out, size_t batch)
{
    if (!ctx) return NB_EINVAL;
    if (batch == 0) return NB_OK;
    if (!in || !out) return fail(ctx, NB_EINVAL, "nb_ntt_forward_i32: null argument");
    NB_ON_DEVICE(ctx);
    NvtxRange nvtx_range("nufhe_b200:ntt_forward");
    ntt_forward_kernel<true><<<ntt_grid(ctx, batch), NTT_SWEEP_THREADS, ntt_smem_bytes(NTT_RAW_I32_BYTES), ctx->stream>>>(in, (u64 *)out, ctx->d_ph_fwd, batch);
    return launch_check(ctx, "ntt_forward_kernel<i32>");
}

int nb_ntt_forward_u64(nb_ctx *ctx, const uint64_t *in, uint64_t *out, size_t batch)
{
    if (!ctx) return NB_EINVAL;
    if (batch == 0) return NB_OK;
    if (!in || !out) return fail(ctx, NB_EINVAL, "nb_ntt_forward_u64: null argument");
    NB_ON_DEVICE(ctx);
    NvtxRange nvtx_range("nufhe_b200:ntt_forward");
    ntt_forward_kernel<false><<<ntt_grid(ctx, batch), NTT_SWEEP_THREADS, ntt_smem_bytes(NTT_RAW_U64_BYTES), ctx->stream>>>(in, (u64 *)out, ctx->d_ph_fwd, batch);
    return launch_check(ctx, "ntt_forward_kernel<u64>");
}

int nb_ntt_inverse_i32(nb_ctx *ctx, const uint64_t *in, int32_t *out, size_t batch)
{
    if (!ctx) return NB_EINVAL;
    if (batch == 0) return NB_OK;
    if (!in || !out) return fail(ctx, NB_EINVAL, "nb_ntt_inverse_i32: null argument");
    NB_ON_DEVICE(ctx);
    NvtxRange nvtx_range("nufhe_b200:ntt_inverse");
    ntt_inverse_kernel<true><<<ntt_grid(ctx, batch), NTT_SWEEP_THREADS, ntt_smem_bytes(NTT_RAW_U64_BYTES), ctx->stream>>>((const u64 *)in, out, ctx->d_ph_inv, batch);
    return launch_check(ctx, "ntt_inverse_kernel<i32>");
}

int nb_ntt_inverse_u64(nb_ctx *ctx, const uint64_t *in, uint64_t *out, size_t batch)
{
    if (!ctx) return NB_EINVAL;
    if (batch == 0) return NB_OK;
    if (!in || !out) return fail(ctx, NB_EINVAL, "nb_ntt_inverse_u64: null argument");
    NB_ON_DEVICE(ctx);
    NvtxRange nvtx_range("nufhe_b200:ntt_inverse");
    ntt_inverse_kernel<false><<<ntt_grid(ctx, batch), NTT_SWEEP_THREADS, ntt_smem_bytes(NTT_RAW_U64_BYTES), ctx->stream>>>((const u64 *)in, out, ctx->d_ph_inv, batch);
    return launch_check(ctx, "ntt_inverse_kernel<u64>");
}

int nb_ff_elementwise(nb_ctx *ctx, int op, const uint64_t *a, const uint64_t *b, uint64_t *out, size_t n,
                      size_t b_period)
{
    if (!ctx || !a || !out) return fail(ctx, NB_EINVAL, "nb_ff_elementwise: null argument");
    if (op < 0 || op > NB_FF_LSH_CONST) return fail(ctx, NB_EINVAL, "nb_ff_elementwise: unknown op");
    if (op != NB_FF_PREPARE && !b) return fail(ctx, NB_EINVAL, "nb_ff_elementwise: binary op needs b");
    if (n == 0) return NB_OK;
    NB_ON_DEVICE(ctx);
    size_t blocks = (n + 255) / 256, cap = (size_t)ctx->sm_count * 16;
    ff_elementwise_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, ctx->stream>>>(
        op, (const u64 *)a, (const u64 *)b, (u64 *)out, n, b_period);
    return launch_check(ctx, "ff_elementwise_kernel");
}

// per key row: the NTT planes (BK_ROW_U64) and the FFT spectra (FFT_ROW_U64).  A key of `rows` rows is laid out as
// all NTT rows first, then all spectra rows (the FFT kernel finds them after n NTT rows).
size_t nb_bk_row_u64(void) { return BK_ROW_U64 + FFT_ROW_U64; }

#ifdef NB_FFT_PHASE_CLOCKS
// profiling builds only (tools/fft_phases.py): copy the per-CTA phase clocks of blind_rotate_fft_kernel
// (fft_kernels.cuh, FFT_CLK_CTAS x FFT_CLK_SLOTS u64) to `out` and, if `reset`, zero them on the device
int nb_fft_phase_clocks(nb_ctx *ctx, unsigned long long *out, int reset)
{
    if (!ctx || !out) return fail(ctx, NB_EINVAL, "nb_fft_phase_clocks: null argument");
    NB_ON_DEVICE(ctx);
    NB_TRY(check(ctx, cudaStreamSynchronize(ctx->stream), "cudaStreamSynchronize"));
    NB_TRY(check(ctx, cudaMemcpyFromSymbol(out, g_fft_phase_clocks, sizeof(g_fft_phase_clocks)), "cudaMemcpyFromSymbol"));
    if (!reset) return NB_OK;
    void *d = nullptr;
    NB_TRY(check(ctx, cudaGetSymbolAddress(&d, g_fft_phase_clocks), "cudaGetSymbolAddress"));
    NB_TRY(check(ctx, cudaMemset(d, 0, sizeof(g_fft_phase_clocks)), "cudaMemset"));
    return check(ctx, cudaDeviceSynchronize(), "cudaDeviceSynchronize");
}
#endif

int nb_bk_prepare(nb_ctx *ctx, const uint64_t *bk_ref, uint64_t *bk_int, size_t rows)
{
    if (!ctx || !bk_ref || !bk_int) return fail(ctx, NB_EINVAL, "nb_bk_prepare: null argument");
    if (rows == 0) return NB_OK;
    NB_ON_DEVICE(ctx);
    NvtxRange nvtx_range("nufhe_b200:bk_prepare");
    size_t total = rows * NTT_N, blocks = (total + 255) / 256, cap = (size_t)ctx->sm_count * 16;
    bk_prepare_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, ctx->stream>>>((const u64 *)bk_ref, (u64 *)bk_int,
                                                                                  ctx->d_ones512, rows);
    NB_TRY(launch_check(ctx, "bk_prepare_kernel"));
    // the key spectra of the FFT kernel: exact int32 coefficients by the inverse transform of the reference key, split
    // into two 16-bit limbs, folded, twisted, transformed and scaled by 1/512 (br_fft.cuh)
    const size_t polys = rows * 8;
    u64 *plain = nullptr;
    i32 *coef = nullptr;
    NB_TRY(check(ctx, cudaMallocAsync((void **)&plain, polys * NTT_N * sizeof(u64), ctx->stream), "cudaMallocAsync"));
    NB_TRY(check(ctx, cudaMallocAsync((void **)&coef, polys * NTT_N * sizeof(i32), ctx->stream), "cudaMallocAsync"));
    blocks = (polys * NTT_N + 255) / 256;
    bk_plain_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, ctx->stream>>>((const u64 *)bk_ref, plain, polys * NTT_N);
    ntt_inverse_kernel<true><<<ntt_grid(ctx, polys), NTT_SWEEP_THREADS, ntt_smem_bytes(NTT_RAW_U64_BYTES), ctx->stream>>>(plain, coef, ctx->d_ph_inv, polys);
    fft_key_kernel<<<(unsigned)(polys * 2), 64, 0, ctx->stream>>>(coef, reinterpret_cast<cplx *>((u64 *)bk_int + rows * BK_ROW_U64), ctx->d_fft_tab);
    NB_TRY(launch_check(ctx, "fft_key_kernel"));
    NB_TRY(check(ctx, cudaFreeAsync(plain, ctx->stream), "cudaFreeAsync"));
    return check(ctx, cudaFreeAsync(coef, ctx->stream), "cudaFreeAsync");
}

}  // extern "C"

// Chunks per chain for `chains` chains on `slots` resident CTAs (kernels.cuh: blind_rotate_kernel).  One wave or
// less needs no slicing.  Otherwise the launch takes ceil(chains * C / slots) rounds of ceil(n / C) steps; each chunk
// also pays for parking / fetching the accumulators (measured: below the noise, profiles/r2_variants.md; 0.1 step here).
static int pick_chunks(size_t chains, size_t slots, int n, int max_chunks)
{
    if (chains <= slots || n <= 1 || max_chunks <= 1) return 1;
    int best = 1;
    double best_cost = 0;
    for (int c = 1; c <= max_chunks && c <= n / 8; c++) {
        const int steps = (n + c - 1) / c;
        const int chunks = (n + steps - 1) / steps;
        const double rounds = (double)((chains * (size_t)chunks + slots - 1) / slots);
        const double cost = rounds * (steps + 0.1);
        if (c == 1 || cost < best_cost * 0.995) { best = chunks; best_cost = cost; }
    }
    return best;
}

static int reserve_words(nb_ctx *ctx, void **buf, size_t *have, size_t want, size_t elem)
{
    if (*have >= want) return NB_OK;
    if (*buf) NB_TRY(check(ctx, cudaFree(*buf), "cudaFree"));
    *buf = nullptr; *have = 0;
    const size_t grow = want + want / 4;
    NB_TRY(check(ctx, cudaMalloc(buf, grow * elem), "cudaMalloc(work queue)"));
    *have = grow;
    return NB_OK;
}

template <class Cfg> static int launch_br_cfg(nb_ctx *ctx, BlindRotateArgs &p)
{
    const size_t slots = (size_t)ctx->sm_count * Cfg::CTAS_PER_SM;
    const size_t chains = (p.batch + Cfg::CT - 1) / Cfg::CT;
    int chunks = p.plain ? 1 : pick_chunks(chains, slots, p.n, ctx->max_chunks);
    if (!p.plain && ctx->force_chunks > 0 && chains > slots) chunks = ctx->force_chunks < p.n ? ctx->force_chunks : p.n;
    p.chains = (unsigned)chains;
    p.steps_per_chunk = p.plain ? 1 : (p.n + chunks - 1) / chunks;
    chunks = p.plain ? 1 : (p.n + p.steps_per_chunk - 1) / p.steps_per_chunk;
    p.chunks = (unsigned)chunks;
    p.sched = nullptr; p.state = nullptr;
    p.sm_count = ctx->sm_count; p.stagger_cycles = ctx->stagger_cycles;
    size_t grid = chains;
    if (chains > slots) {
        // more than one wave: persistent CTAs pull (chain, chunk) tickets
        // ready queue: head, tail, then one entry per (chain, chunk); entries of first chunks stay 0 (implicit)
        const size_t entries = chunks > 1 ? chains * (size_t)chunks : 0;
        NB_TRY(reserve_words(ctx, (void **)&ctx->d_sched, &ctx->sched_words, BR_SCHED_HEADER + entries, sizeof(unsigned)));
        if (chunks > 1)
            NB_TRY(reserve_words(ctx, (void **)&ctx->d_state, &ctx->state_words, chains * Cfg::CT * 2 * NTT_N, sizeof(int32_t)));
        NB_TRY(check(ctx, cudaMemsetAsync(ctx->d_sched, 0, (BR_SCHED_HEADER + entries) * sizeof(unsigned), ctx->stream), "cudaMemsetAsync"));
        p.sched = ctx->d_sched; p.state = ctx->d_state;
        grid = slots;
    }
    if constexpr (std::is_same_v<Cfg, BrFft>)
        blind_rotate_fft_kernel<Cfg><<<(int)grid, Cfg::THREADS, br_fft_smem_bytes<Cfg>(), ctx->stream>>>(p, ctx->d_fft_tab);
    else
        blind_rotate_kernel<Cfg><<<(int)grid, Cfg::THREADS, br_smem_bytes<Cfg>(), ctx->stream>>>(p, ctx->d_ph_fwd, ctx->d_ph_inv);
    return NB_OK;
}

// One launch of the fused kernel in the shape that suits the batch: "wide" CTAs (1 ciphertext on 256 threads,
// shortest step) while the batch fits one wave of them, else 2 ciphertexts per CTA (highest throughput).
static int launch_br(nb_ctx *ctx, BlindRotateArgs &p)
{
    if (!p.plain && p.n > 0 && p.batch <= ctx->pair_max) {
        p.sched = nullptr; p.state = nullptr; p.chains = (unsigned)p.batch; p.chunks = 1; p.steps_per_chunk = p.n;
        p.sm_count = ctx->sm_count; p.stagger_cycles = 0;
        if (ctx->pair_async) blind_rotate_pair_kernel<true><<<(unsigned)(2 * p.batch), PAIR_THREADS, BR_PAIR_SMEM_BYTES, ctx->stream>>>(p, ctx->d_ph_fwd, ctx->d_ph_inv);
        else blind_rotate_pair_kernel<false><<<(unsigned)(2 * p.batch), PAIR_THREADS, BR_PAIR_SMEM_BYTES, ctx->stream>>>(p, ctx->d_ph_fwd, ctx->d_ph_inv);
        return NB_OK;
    }
    if (p.batch <= ctx->wide2_max) return launch_br_cfg<BrWide2>(ctx, p);
    if (p.batch <= ctx->wide_max) return launch_br_cfg<BrWide>(ctx, p);
    // gate bootstraps (the key handle then has exactly n rows, so the spectra follow the n NTT rows)
    if (ctx->use_fft && !p.plain && !p.bara && p.n > 0) return launch_br_cfg<BrFft>(ctx, p);
    return launch_br_cfg<BrDefault>(ctx, p);
}

extern "C" {

int nb_ctx_reserve(nb_ctx *ctx, size_t batch)
{
    if (!ctx) return NB_EINVAL;
    NB_ON_DEVICE(ctx);
    // everything launch_br_cfg / nb_keyswitch could ask for with up to `batch` ciphertexts (2 * batch for gate_mux's
    // double launch is the caller's business): after this, those calls never allocate, so they can be captured
    NB_TRY(reserve_words(ctx, (void **)&ctx->d_sched, &ctx->sched_words, BR_SCHED_HEADER + (batch + 1) * (size_t)ctx->max_chunks, sizeof(unsigned)));
    NB_TRY(reserve_words(ctx, (void **)&ctx->d_state, &ctx->state_words, (batch + 2) * 2 * NTT_N, sizeof(int32_t)));
    NB_TRY(reserve_words(ctx, (void **)&ctx->d_cv_blocks, &ctx->cv_words, batch * KS_CV_BLOCKS, sizeof(float)));
    return NB_OK;
}

int nb_external_product(nb_ctx *ctx, int32_t *accum, const uint64_t *bk_int, size_t bk_row, size_t batch)
{
    if (ctx && batch == 0) return NB_OK;     // nothing to do: empty arrays have no storage to check
    if (!ctx || !accum || !bk_int) return fail(ctx, NB_EINVAL, "nb_external_product: null argument");
    if (batch == 0) return NB_OK;
    NB_ON_DEVICE(ctx);
    NvtxRange nvtx_range("nufhe_b200:external_product");
    BlindRotateArgs p{};
    p.accum = accum; p.accum_out = accum; p.bk = (const u64 *)bk_int + bk_row * BK_ROW_U64;
    p.plain = 1; p.batch = batch;
    NB_TRY(launch_br(ctx, p));
    return launch_check(ctx, "blind_rotate_kernel(plain external product)");
}

static int launch_blind_rotate(nb_ctx *ctx, BlindRotateArgs &p)
{
    if (p.n <= 0 || p.n > LWE_N_MAX) return fail(ctx, NB_EUNSUPPORTED, "LWE dimension out of range");
    if (p.batch == 0) return NB_OK;
    NB_ON_DEVICE(ctx);
    NvtxRange nvtx_range("nufhe_b200:gate_prologue+blind_rotate+extract");
    NB_TRY(launch_br(ctx, p));
    return launch_check(ctx, "blind_rotate_kernel");
}

int nb_blind_rotate(nb_ctx *ctx, const int32_t *accum, const int32_t *bara, const uint64_t *bk_int, size_t n,
                    int32_t *out_a, int32_t *out_b, int32_t *accum_out, size_t batch)
{
    if (ctx && batch == 0) return NB_OK;     // nothing to do: empty arrays have no storage to check
    if (!ctx || !accum || !bara || !bk_int) return fail(ctx, NB_EINVAL, "nb_blind_rotate: null argument");
    if ((out_a == nullptr) != (out_b == nullptr)) return fail(ctx, NB_EINVAL, "nb_blind_rotate: out_a/out_b must come together");
    BlindRotateArgs p{};
    p.accum = accum; p.bara = bara; p.bk = (const u64 *)bk_int; p.n = (int)n;
    p.out_a = out_a; p.out_b = out_b; p.accum_out = accum_out; p.extract = out_a != nullptr; p.batch = batch;
    return launch_blind_rotate(ctx, p);
}

int nb_bootstrap_extract(nb_ctx *ctx, const int32_t *in1_a, const int32_t *in1_b, const int32_t *in2_a,
                         const int32_t *in2_b, int32_t c, int32_t s1, int32_t s2, int32_t mu,
                         const uint64_t *bk_int, size_t n, int32_t *out_a, int32_t *out_b, size_t batch)
{
    if (ctx && batch == 0) return NB_OK;     // nothing to do: empty arrays have no storage to check
    if (!ctx || !in1_a || !in1_b || !bk_int || !out_a || !out_b)
        return fail(ctx, NB_EINVAL, "nb_bootstrap_extract: null argument");
    if ((in2_a == nullptr) != (in2_b == nullptr)) return fail(ctx, NB_EINVAL, "nb_bootstrap_extract: in2_a/in2_b must come together");
    BlindRotateArgs p{};
    p.in1_a = in1_a; p.in1_b = in1_b; p.in2_a = in2_a; p.in2_b = in2_b;
    p.c = c; p.s1 = s1; p.s2 = s2; p.mu = mu;
    p.bk = (const u64 *)bk_int; p.n = (int)n; p.out_a = out_a; p.out_b = out_b; p.extract = 1; p.batch = batch;
    return launch_blind_rotate(ctx, p);
}

int nb_bootstrap_extract2(nb_ctx *ctx, const int32_t *a1_a, const int32_t *a1_b, const int32_t *a2_a,
                          const int32_t *a2_b, int32_t a_c, int32_t a_s1, int32_t a_s2, const int32_t *b1_a,
                          const int32_t *b1_b, const int32_t *b2_a, const int32_t *b2_b, int32_t b_c, int32_t b_s1,
                          int32_t b_s2, int32_t mu, const uint64_t *bk_int, size_t n, int32_t *out_a, int32_t *out_b,
                          size_t batch)
{
    if (ctx && batch == 0) return NB_OK;     // nothing to do: empty arrays have no storage to check
    if (!ctx || !a1_a || !a1_b || !b1_a || !b1_b || !bk_int || !out_a || !out_b)
        return fail(ctx, NB_EINVAL, "nb_bootstrap_extract2: null argument");
    if ((a2_a == nullptr) != (a2_b == nullptr) || (b2_a == nullptr) != (b2_b == nullptr))
        return fail(ctx, NB_EINVAL, "nb_bootstrap_extract2: a/b parts must come together");
    BlindRotateArgs p{};
    p.in1_a = a1_a; p.in1_b = a1_b; p.in2_a = a2_a; p.in2_b = a2_b; p.c = a_c; p.s1 = a_s1; p.s2 = a_s2;
    p.j2_in1_a = b1_a; p.j2_in1_b = b1_b; p.j2_in2_a = b2_a; p.j2_in2_b = b2_b; p.j2_c = b_c; p.j2_s1 = b_s1; p.j2_s2 = b_s2;
    p.mu = mu; p.job_batch = batch;
    p.bk = (const u64 *)bk_int; p.n = (int)n; p.out_a = out_a; p.out_b = out_b; p.extract = 1; p.batch = 2 * batch;
    return launch_blind_rotate(ctx, p);
}

int nb_keyswitch(nb_ctx *ctx, const int32_t *src1_a, const int32_t *src1_b, const int32_t *src2_a,
                 const int32_t *src2_b, int32_t c, const int32_t *ks_a, const int32_t *ks_b, const float *ks_cv,
                 size_t in_size, size_t n, int t, int log2_base, int32_t *res_a, int32_t *res_b, float *res_cv,
                 size_t batch)
{
    if (ctx && batch == 0) return NB_OK;     // nothing to do: empty arrays have no storage to check
    if (!ctx || !src1_a || !src1_b || !ks_a || !ks_b || !ks_cv || !res_a || !res_b)
        return fail(ctx, NB_EINVAL, "nb_keyswitch: null argument");
    if ((src2_a == nullptr) != (src2_b == nullptr)) return fail(ctx, NB_EINVAL, "nb_keyswitch: src2_a/src2_b must come together");
    if (n + 1 > 512) return fail(ctx, NB_EUNSUPPORTED, "nb_keyswitch: output LWE dimension above 511");
    if (t < 1 || log2_base < 1 || t * log2_base > 31) return fail(ctx, NB_EINVAL, "nb_keyswitch: bad decomposition");
    if (batch == 0) return NB_OK;
    NB_ON_DEVICE(ctx);
    NvtxRange nvtx_range("nufhe_b200:keyswitch");
    KeyswitchArgs p{};
    p.src1_a = src1_a; p.src1_b = src1_b; p.src2_a = src2_a; p.src2_b = src2_b; p.c = c;
    p.ks_a = ks_a; p.ks_b = ks_b; p.ks_cv = ks_cv; p.res_a = res_a; p.res_b = res_b; p.res_cv = res_cv;
    p.in_size = (int)in_size; p.n = (int)n; p.t = t; p.log2_base = log2_base; p.batch = batch;
    if (t == 8 && log2_base == 2 && in_size == (size_t)KS_IN && n == (size_t)KS_N) {
        // The consumer loop always walks KS_TILE ciphertext slots, so a CTA costs the same whatever its tile:
        // fill the tiles, then split the 1024 input coefficients over blockIdx.y until the SMs are covered
        // (partial sums meet in integer atomics).  One ciphertext: 128 CTAs x 8 coefficients.
        size_t tile = batch < (size_t)KS_TILE ? batch : (size_t)KS_TILE;
        p.tile = (int)tile;
        int grid = (int)((batch + tile - 1) / tile);
        int splits = ctx->sm_count / grid;
        if (splits > 128) splits = 128;
        if (splits < 1) splits = 1;
        p.splits = splits;
        if (splits > 1) {
            NB_TRY(check(ctx, cudaMemsetAsync(res_a, 0, batch * n * sizeof(int32_t), ctx->stream), "cudaMemsetAsync"));
            NB_TRY(check(ctx, cudaMemsetAsync(res_b, 0, batch * sizeof(int32_t), ctx->stream), "cudaMemsetAsync"));
        }
        if (splits > 1 && res_cv) {
            NB_TRY(reserve_words(ctx, (void **)&ctx->d_cv_blocks, &ctx->cv_words, batch * KS_CV_BLOCKS, sizeof(float)));
            p.cv_blocks = ctx->d_cv_blocks;
        }
        keyswitch_kernel<<<dim3(grid, splits), KS_THREADS, KS_SMEM_BYTES, ctx->stream>>>(p);
        if (p.cv_blocks) {
            NB_TRY(launch_check(ctx, "keyswitch_kernel"));
            ks_cv_finalize_kernel<<<(int)((batch + 127) / 128), 128, 0, ctx->stream>>>(res_cv, p.cv_blocks, batch);
        }
    } else {
        keyswitch_generic_kernel<<<(int)batch, 512, 0, ctx->stream>>>(p);
    }
    return launch_check(ctx, "keyswitch_kernel");
}

static int ew_grid(nb_ctx *ctx, size_t n)
{
    size_t blocks = (n + 255) / 256, cap = (size_t)ctx->sm_count * 16;
    return (int)(blocks < cap ? blocks : cap);
}

int nb_shift_torus_polynomial(nb_ctx *ctx, int32_t *result, const int32_t *source, const int32_t *powers,
                              size_t powers_stride, size_t power_idx, int polys_per_power, int mode, int n_log2,
                              size_t polys)
{
    if (!ctx) return NB_EINVAL;
    if (!result || !source || !powers) return fail(ctx, NB_EINVAL, "nb_shift_torus_polynomial: null argument");
    if (mode < NB_SHIFT_INVERT || mode > NB_SHIFT_PLAIN) return fail(ctx, NB_EINVAL, "nb_shift_torus_polynomial: unknown mode");
    if (n_log2 < 1 || n_log2 > 20 || polys_per_power < 1) return fail(ctx, NB_EINVAL, "nb_shift_torus_polynomial: bad size");
    if (result == source) return fail(ctx, NB_EINVAL, "nb_shift_torus_polynomial: result must not alias source");
    if (polys == 0) return NB_OK;
    NB_ON_DEVICE(ctx);
    shift_torus_polynomial_kernel<<<ew_grid(ctx, polys << n_log2), 256, 0, ctx->stream>>>(
        result, source, powers, powers_stride, power_idx, polys_per_power, mode, n_log2, polys);
    return launch_check(ctx, "shift_torus_polynomial_kernel");
}

int nb_tlwe_noiseless_trivial(nb_ctx *ctx, int32_t *acc, float *cv, const int32_t *mu, int mask_size, int n_log2,
                              size_t batch)
{
    if (!ctx) return NB_EINVAL;
    if (!acc || !mu) return fail(ctx, NB_EINVAL, "nb_tlwe_noiseless_trivial: null argument");
    if (mask_size < 1 || n_log2 < 1 || n_log2 > 20) return fail(ctx, NB_EINVAL, "nb_tlwe_noiseless_trivial: bad size");
    if (batch == 0) return NB_OK;
    NB_ON_DEVICE(ctx);
    tlwe_noiseless_trivial_kernel<<<ew_grid(ctx, (batch * (mask_size + 1)) << n_log2), 256, 0, ctx->stream>>>(
        acc, cv, mu, mask_size, n_log2, batch);
    return launch_check(ctx, "tlwe_noiseless_trivial_kernel");
}

int nb_tlwe_extract_lwe_samples(nb_ctx *ctx, int32_t *out_a, int32_t *out_b, const int32_t *acc, int mask_size,
                                int n_log2, size_t batch)
{
    if (!ctx) return NB_EINVAL;
    if (!out_a || !out_b || !acc) return fail(ctx, NB_EINVAL, "nb_tlwe_extract_lwe_samples: null argument");
    if (mask_size < 1 || n_log2 < 1 || n_log2 > 20) return fail(ctx, NB_EINVAL, "nb_tlwe_extract_lwe_samples: bad size");
    if (batch == 0) return NB_OK;
    NB_ON_DEVICE(ctx);
    tlwe_extract_lwe_samples_kernel<<<ew_grid(ctx, (batch * mask_size) << n_log2), 256, 0, ctx->stream>>>(
        out_a, out_b, acc, mask_size, n_log2, batch);
    return launch_check(ctx, "tlwe_extract_lwe_samples_kernel");
}

int nb_t32_to_phase(nb_ctx *ctx, int32_t *out, const int32_t *in, size_t n, uint32_t mspace_size)
{
    if (!ctx) return NB_EINVAL;
    if (!out || !in) return fail(ctx, NB_EINVAL, "nb_t32_to_phase: null argument");
    if (mspace_size == 0 || (mspace_size & (mspace_size - 1))) return fail(ctx, NB_EINVAL, "nb_t32_to_phase: mspace_size must be a power of two");
    if (n == 0) return NB_OK;
    NB_ON_DEVICE(ctx);
    t32_to_phase_kernel<<<ew_grid(ctx, n), 256, 0, ctx->stream>>>(out, in, n, mspace_size);
    return launch_check(ctx, "t32_to_phase_kernel");
}

int nb_tgsw_decompose(nb_ctx *ctx, int32_t *out, const int32_t *in, size_t polys, int decomp_length, int bs_log2_base,
                      int32_t offset, int n_log2)
{
    if (!ctx) return NB_EINVAL;
    if (!out || !in) return fail(ctx, NB_EINVAL, "nb_tgsw_decompose: null argument");
    if (decomp_length < 1 || bs_log2_base < 1 || decomp_length * bs_log2_base > 32 || n_log2 < 1 || n_log2 > 20)
        return fail(ctx, NB_EINVAL, "nb_tgsw_decompose: bad decomposition");
    if (polys == 0) return NB_OK;
    NB_ON_DEVICE(ctx);
    tgsw_decompose_kernel<<<ew_grid(ctx, (polys * decomp_length) << n_log2), 256, 0, ctx->stream>>>(
        out, in, polys, decomp_length, bs_log2_base, offset, n_log2);
    return launch_check(ctx, "tgsw_decompose_kernel");
}

int nb_tgsw_mac(nb_ctx *ctx, uint64_t *out, const uint64_t *tr, const uint64_t *bk_row, size_t batch, int mask_size,
                int decomp_length)
{
    if (!ctx) return NB_EINVAL;
    if (!out || !tr || !bk_row) return fail(ctx, NB_EINVAL, "nb_tgsw_mac: null argument");
    if (mask_size < 1 || mask_size > 15 || decomp_length < 1 || decomp_length > 32) return fail(ctx, NB_EINVAL, "nb_tgsw_mac: bad size");
    if (batch == 0) return NB_OK;
    NB_ON_DEVICE(ctx);
    tgsw_mac_kernel<<<ew_grid(ctx, batch * (mask_size + 1) * NTT_N), 256, 0, ctx->stream>>>(
        (u64 *)out, (const u64 *)tr, (const u64 *)bk_row, batch, mask_size + 1, decomp_length);
    return launch_check(ctx, "tgsw_mac_kernel");
}

int nb_tlwe_add_to(nb_ctx *ctx, int32_t *res, const int32_t *src, size_t n, float *res_cv, const float *src_cv,
                   size_t n_cv)
{
    if (!ctx) return NB_EINVAL;
    if (!res || !src || ((res_cv == nullptr) != (src_cv == nullptr)))
        return fail(ctx, NB_EINVAL, "nb_tlwe_add_to: null argument");
    if (n_cv > n) return fail(ctx, NB_EINVAL, "nb_tlwe_add_to: more variances than coefficients");
    if (n == 0) return NB_OK;
    NB_ON_DEVICE(ctx);
    add_to_kernel<<<ew_grid(ctx, n), 256, 0, ctx->stream>>>(res, src, n, res_cv, src_cv, res_cv ? n_cv : 0);
    return launch_check(ctx, "add_to_kernel");
}

int nb_lwe_affine(nb_ctx *ctx, int32_t *res_a, int32_t *res_b, const int32_t *x1_a, const int32_t *x1_b,
                  const int32_t *x2_a, const int32_t *x2_b, int32_t c, int32_t s1, int32_t s2, size_t batch,
                  size_t n)
{
    if (ctx && batch == 0) return NB_OK;     // nothing to do: empty arrays have no storage to check
    if (!ctx || !res_a || !res_b) return fail(ctx, NB_EINVAL, "nb_lwe_affine: null argument");
    if ((x1_a == nullptr) != (x1_b == nullptr) || (x2_a == nullptr) != (x2_b == nullptr))
        return fail(ctx, NB_EINVAL, "nb_lwe_affine: a/b parts must come together");
    if (batch == 0) return NB_OK;
    NB_ON_DEVICE(ctx);
    size_t total = batch * (n + 1), blocks = (total + 255) / 256, cap = (size_t)ctx->sm_count * 16;
    lwe_affine_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, ctx->stream>>>(
        res_a, res_b, x1_a, x1_b, x2_a, x2_b, c, s1, s2, batch, (int)n);
    return launch_check(ctx, "lwe_affine_kernel");
}

int nb_lwe_dot(nb_ctx *ctx, int32_t *out, const int32_t *a, const int32_t *key, const int32_t *add1,
               const int32_t *add2, int32_t sign, size_t batch, size_t n)
{
    if (!ctx) return NB_EINVAL;
    if (batch == 0) return NB_OK;
    if (!out || !a || !key) return fail(ctx, NB_EINVAL, "nb_lwe_dot: null argument");
    if (n == 0 || n > (1u << 30)) return fail(ctx, NB_EINVAL, "nb_lwe_dot: bad LWE dimension");
    if (batch == 0) return NB_OK;
    NB_ON_DEVICE(ctx);
    NvtxRange nvtx_range("nufhe_b200:lwe_dot");
    size_t blocks = (batch * 32 + 255) / 256, cap = (size_t)ctx->sm_count * 16;
    lwe_dot_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, ctx->stream>>>(out, a, key, add1, add2, sign, batch, (int)n);
    return launch_check(ctx, "lwe_dot_kernel");
}

int nb_make_keyswitch_key(nb_ctx *ctx, int32_t *ks_a, int32_t *ks_b, float *ks_cv, const int32_t *in_key,
                          const int32_t *out_key, const int32_t *noises_a, const int32_t *noises_b, size_t in_size,
                          size_t n, int t, int log2_base, float noise_variance)
{
    if (!ctx) return NB_EINVAL;
    if (!ks_a || !ks_b || !ks_cv || !in_key || !out_key || !noises_a || !noises_b)
        return fail(ctx, NB_EINVAL, "nb_make_keyswitch_key: null argument");
    if (t < 1 || log2_base < 1 || t * log2_base > 31 || n == 0) return fail(ctx, NB_EINVAL, "nb_make_keyswitch_key: bad decomposition");
    if (in_size == 0) return NB_OK;
    NB_ON_DEVICE(ctx);
    NvtxRange nvtx_range("nufhe_b200:make_keyswitch_key");
    const size_t rows = in_size * (size_t)t << log2_base;
    size_t blocks = (rows * 32 + 255) / 256, cap = (size_t)ctx->sm_count * 16;
    make_keyswitch_key_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, ctx->stream>>>(
        ks_a, ks_b, ks_cv, in_key, out_key, noises_a, noises_b, in_size, (int)n, t, log2_base, noise_variance);
    return launch_check(ctx, "make_keyswitch_key_kernel");
}

}  // extern "C"
