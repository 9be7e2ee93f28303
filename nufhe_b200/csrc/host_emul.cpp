// host_emul.cpp -- runs the __host__ __device__ pass code of br_phases.cuh / ntt_lane.cuh on the CPU, one
// "thread" after the other, a phase at a time (a phase boundary = a CTA barrier).  Built with g++ into
// libnb_host_emul.so for tests/test_host_logic.py: it lets the CPU-only test suite check the index maps,
// swizzles, twiddle tables and shift constants of the GPU kernels against the oracle.
// This is a test aid for the CUDA source, not a CPU fallback: nothing in nufhe_b200/ loads it.
#include <cstring>
#include <vector>
#include "tables.h"

using namespace nb;

extern "C" {

// The stand-alone transform kernels' passes, one polynomial at a time; in/out natural order, canonical.
void emul_ntt_forward(const u64 *in, u64 *out, size_t batch)
{
    static PhaseTables T;
    std::vector<u64> w(NTT_SWEEP_POLYS * POLY_STRIDE);
    for (size_t b = 0; b < batch; b++) {
        for (int task = 0; task < 64; task++) {
            u64 x[16];
            for (int j1 = 0; j1 < 16; j1++) x[j1] = ff_canon(in[b * NTT_N + 64 * j1 + task]);
            phase_fwd1_generic(task, x, w.data(), T.fwd.data());
        }
        for (int row = 0; row < 16; row++) for (int g = 0; g < 4; g++) phase_fwd2(0, row, g, w.data());
        for (int row = 0; row < 16; row++) for (int u = 0; u < 4; u++) phase_fwd3(0, row, u, w.data());
        for (int k = 0; k < NTT_N; k++) out[b * NTT_N + k] = ff_canon(w[w_position_of_natural(k)]);
    }
}

void emul_ntt_inverse(const u64 *in, u64 *out, size_t batch)
{
    static PhaseTables T;
    std::vector<u64> w(NTT_SWEEP_POLYS * POLY_STRIDE);
    for (size_t b = 0; b < batch; b++) {
        for (int k = 0; k < NTT_N; k++) w[w_position_of_natural(k)] = ff_canon(in[b * NTT_N + k]);
        for (int row = 0; row < 16; row++) for (int u = 0; u < 4; u++) phase_inv3(0, row, u, w.data());
        for (int row = 0; row < 16; row++) for (int g = 0; g < 4; g++) phase_inv2(0, row, g, w.data());
        for (int task = 0; task < 64; task++) {
            u64 y[16];
            phase_inv1_generic(task, y, w.data(), T.inv.data());
            for (int j1 = 0; j1 < 16; j1++) out[b * NTT_N + 64 * j1 + task] = ff_canon(y[j1]);
        }
    }
}

// the same with Torus32 on the natural-order side (i32_conversion): forward reads int32, inverse writes int32
void emul_ntt_forward_i32(const i32 *in, u64 *out, size_t batch)
{
    static PhaseTables T;
    std::vector<u64> w(NTT_SWEEP_POLYS * POLY_STRIDE);
    for (size_t b = 0; b < batch; b++) {
        for (int task = 0; task < 64; task++) {
            i32 x[16];
            for (int j1 = 0; j1 < 16; j1++) x[j1] = in[b * NTT_N + 64 * j1 + task];
            phase_fwd1_i32(task, x, w.data(), T.fwd.data());
        }
        for (int row = 0; row < 16; row++) for (int g = 0; g < 4; g++) phase_fwd2(0, row, g, w.data());
        for (int row = 0; row < 16; row++) for (int u = 0; u < 4; u++) phase_fwd3(0, row, u, w.data());
        for (int k = 0; k < NTT_N; k++) out[b * NTT_N + k] = ff_canon(w[w_position_of_natural(k)]);
    }
}

void emul_ntt_inverse_i32(const u64 *in, i32 *out, size_t batch)
{
    static PhaseTables T;
    std::vector<u64> w(NTT_SWEEP_POLYS * POLY_STRIDE);
    for (size_t b = 0; b < batch; b++) {
        for (int k = 0; k < NTT_N; k++) w[w_position_of_natural(k)] = ff_canon(in[b * NTT_N + k]);
        for (int row = 0; row < 16; row++) for (int u = 0; u < 4; u++) phase_inv3(0, row, u, w.data());
        for (int row = 0; row < 16; row++) for (int g = 0; g < 4; g++) phase_inv2(0, row, g, w.data());
        for (int task = 0; task < 64; task++) {
            i32 y[16];
            phase_inv1_i32(task, y, w.data(), T.inv.data());
            for (int j1 = 0; j1 < 16; j1++) out[b * NTT_N + 64 * j1 + task] = y[j1];
        }
    }
}

// One external-product step of the phase-structured kernel (br_phases.cuh) for up to BR2_CT
// ciphertexts, phases executed in order with all "threads" of a phase run back to back.
// acc: (nct, 2, 1024) in/out; bk_ref_row: reference layout (2,2,2,1024) Montgomery; rot: rotation
// amounts per ciphertext or NULL (plain external product, overwrite).
int emul_phase_ct(void) { return BR2_CT; }

}  // extern "C"

static void prepare_bk_row(const u64 *bk_ref_row, const PhaseTables &T, std::vector<u64> &bk);

template <class Cfg> static void phase_step(i32 *acc_io, const u64 *bk_ref_row, const int *rot, int nct)
{
    static PhaseTables T;
    std::vector<i32> acc(Cfg::CT * 2 * NTT_N, 0);
    std::vector<u64> w(Cfg::POLYS * POLY_STRIDE, 0);
    std::vector<u64> bk(BK_ROW_U64);
    for (int c = 0; c < nct; c++) memcpy(&acc[c * 2 * NTT_N], acc_io + c * 2 * NTT_N, sizeof(i32) * 2 * NTT_N);
    int rots[4] = {0, 0, 0, 0};
    if (rot) for (int c = 0; c < nct; c++) rots[c] = rot[c];
    prepare_bk_row(bk_ref_row, T, bk);
    constexpr int TH = Cfg::THREADS;
    if constexpr (Cfg::SPLIT_FWD) {
        using Tasks = BrCfg<Cfg::CT, 256 * Cfg::CT>;
        auto each = [&](auto fn) { for (int tid = 0; tid < TH; tid++) { int h, t; map_split_fwd<Cfg>(tid, h, t); fn(h, t); } };
        each([&](int h, int t) {
            if (rot) { if (h) phase_fwd1_split<true, 1>(t, acc.data(), w.data(), T.fwd.data(), rots); else phase_fwd1_split<true, 0>(t, acc.data(), w.data(), T.fwd.data(), rots); }
            else { if (h) phase_fwd1_split<false, 1>(t, acc.data(), w.data(), T.fwd.data(), rots); else phase_fwd1_split<false, 0>(t, acc.data(), w.data(), T.fwd.data(), rots); }
        });
        each([&](int h, int t) { int p, r, g; map_fwd2<Tasks>(t, 0, p, r, g); if (h) phase_fwd2_split<1>(p, r, g, w.data()); else phase_fwd2_split<0>(p, r, g, w.data()); });
        {   // in place: every thread holds its 16 inputs in registers across a barrier
            std::vector<u64> held((size_t)TH * 16);
            each([&](int h, int t) { int p, r, u; map_fwd3<Tasks>(t, 0, p, r, u); phase_fwd3_split_load(p, r, u, w.data(), &held[(size_t)(h * 256 * Cfg::CT + t) * 16]); });
            each([&](int h, int t) {
                int p, r, u; map_fwd3<Tasks>(t, 0, p, r, u);
                const u64 *v = &held[(size_t)(h * 256 * Cfg::CT + t) * 16];
                if (h) phase_fwd3_split_finish<1>(p, r, u, w.data(), v); else phase_fwd3_split_finish<0>(p, r, u, w.data(), v);
            });
        }
    } else {
        if constexpr (Cfg::FWD1_BOTH_DIGITS) {
            for (int tid = 0; tid < TH; tid++) {
                if (rot) phase_fwd1_both_digits<true>(tid, acc.data(), w.data(), T.fwd.data(), rots);
                else phase_fwd1_both_digits<false>(tid, acc.data(), w.data(), T.fwd.data(), rots);
            }
        } else {
            for (int it = 0; it < Cfg::FWD_SWEEPS; it++)
                for (int tid = 0; tid < TH; tid++) {
                    if (rot) phase_fwd1<true>(it * TH + tid, acc.data(), w.data(), T.fwd.data(), rots);
                    else phase_fwd1<false>(it * TH + tid, acc.data(), w.data(), T.fwd.data(), rots);
                }
        }
        for (int it = 0; it < Cfg::FWD_SWEEPS; it++)
            for (int tid = 0; tid < TH; tid++) { int p, r, g; map_fwd2<Cfg>(tid, it, p, r, g); phase_fwd2(p, r, g, w.data()); }
        for (int it = 0; it < Cfg::FWD_SWEEPS; it++)
            for (int tid = 0; tid < TH; tid++) { int p, r, u; map_fwd3<Cfg>(tid, it, p, r, u); phase_fwd3(p, r, u, w.data()); }
    }
    for (int tid = 0; tid < TH; tid++) phase_mac<Cfg>(tid, w.data(), bk.data());
    if constexpr (Cfg::SPLIT_INV) {
        // the split inverse phases of the wide shape, one loop per barrier-separated sub-pass (kernels.cuh: br2_step)
        auto each = [&](auto fn) { for (int tid = 0; tid < TH; tid++) { int h, t; if (map_split<Cfg>(tid, h, t)) fn(h, t); } };
        each([&](int h, int t) { int p, r, u; map_inv3<Cfg>(t, p, r, u); if (h) phase_inv3_split_a<1>(p, r, u, w.data()); else phase_inv3_split_a<0>(p, r, u, w.data()); });
        each([&](int h, int t) { int p, r, u; map_inv3<Cfg>(t, p, r, u); if (h) phase_inv3_split_b<1>(p, r, u, w.data()); else phase_inv3_split_b<0>(p, r, u, w.data()); });
        each([&](int h, int t) { int p, r, g; map_inv2_split<Cfg>(t, p, r, g); if (h) phase_inv2_split<1>(p, r, g, w.data()); else phase_inv2_split<0>(p, r, g, w.data()); });
        each([&](int h, int t) { if (h) phase_inv1_split_a<1>(t, w.data(), T.inv.data()); else phase_inv1_split_a<0>(t, w.data(), T.inv.data()); });
        each([&](int h, int t) {
            if (rot) { if (h) phase_inv1_split_b<true, 1>(t, acc.data(), w.data()); else phase_inv1_split_b<true, 0>(t, acc.data(), w.data()); }
            else { if (h) phase_inv1_split_b<false, 1>(t, acc.data(), w.data()); else phase_inv1_split_b<false, 0>(t, acc.data(), w.data()); }
        });
    } else {
        for (int tid = 0; tid < TH; tid++) { int p, r, u; if (map_inv3<Cfg>(tid, p, r, u)) phase_inv3(p, r, u, w.data()); }
        for (int tid = 0; tid < TH; tid++) { int p, r, g; if (map_inv2<Cfg>(tid, p, r, g)) phase_inv2(p, r, g, w.data()); }
        for (int tid = 0; tid < Cfg::INV_TASKS; tid++) {
            if (rot) phase_inv1<true>(tid, acc.data(), w.data(), T.inv.data());
            else phase_inv1<false>(tid, acc.data(), w.data(), T.inv.data());
        }
    }
    for (int c = 0; c < nct; c++) memcpy(acc_io + c * 2 * NTT_N, &acc[c * 2 * NTT_N], sizeof(i32) * 2 * NTT_N);
}

// the engine layout of one reference key row (kernels.cuh: bk_prepare_kernel)
static void prepare_bk_row(const u64 *bk_ref_row, const PhaseTables &T, std::vector<u64> &bk)
{
    bk.assign(BK_ROW_U64, 0);
    for (int pos = 0; pos < NTT_N; pos++) {
        const int k = w_natural_index(pos >> 6, pos & 63);
        u64 sum[2] = {0, 0};
        for (int m = 0; m < 8; m++) {
            u64 x = ff_mul(ff_canon(bk_ref_row[m * NTT_N + k]), FF_RINV);
            bk[m * NTT_N + pos] = x;
            sum[m & 1] = ff_add(sum[m & 1], x);
        }
        for (int mo = 0; mo < 2; mo++) bk[(8 + mo) * NTT_N + pos] = ff_mul(sum[mo], T.ones512[k]);
    }
}

// `steps` consecutive CMux steps of the pair shape (kernels.cuh: blind_rotate_pair_kernel) with the same key row: two
// "CTAs", each with its own work polynomials and accumulator polynomial, every barrier-separated sub-phase run for both
// before the next one starts; the remote stores of the MAC go straight into the other CTA's array.  Several steps in a
// row exercise both parities of the exchange area and what one step leaves behind for the next.
static void pair_steps(i32 *acc_io, const u64 *bk_ref_row, const int *rots, int steps)
{
    static PhaseTables T;
    std::vector<u64> bk;
    prepare_bk_row(bk_ref_row, T, bk);
    std::vector<u64> w[2] = {std::vector<u64>(PAIR_POLYS * POLY_STRIDE, 0x1234567887654321ull), std::vector<u64>(PAIR_POLYS * POLY_STRIDE, 0x0fedcba987654321ull)};
    i32 *acc[2] = {acc_io, acc_io + NTT_N};
    auto both = [&](int threads, auto fn) { for (int rank = 0; rank < 2; rank++) for (int tid = 0; tid < threads; tid++) fn(rank, tid); };
    for (int i = 0; i < steps; i++) {
        const int par = i & 1;
        const int *rot = rots + i;
        both(PAIR_THREADS, [&](int r, int tid) { pair_fwd1(tid, acc[r], w[r].data(), T.fwd.data(), rot); });
        both(PAIR_THREADS, [&](int r, int tid) { pair_fwd2(tid, w[r].data()); });
        std::vector<u64> held((size_t)2 * PAIR_THREADS * 16);
        both(PAIR_THREADS, [&](int r, int tid) { pair_fwd3_load(tid, w[r].data(), &held[((size_t)r * PAIR_THREADS + tid) * 16]); });
        both(PAIR_THREADS, [&](int r, int tid) { pair_fwd3_finish(tid, w[r].data(), &held[((size_t)r * PAIR_THREADS + tid) * 16]); });
        both(PAIR_THREADS, [&](int r, int tid) {
            u64 *peer = w[r ^ 1].data();
            pair_mac<false>(tid, w[r].data(), [peer](int off, u64 x, u64 y) { peer[off] = x; peer[off + 1] = y; },
                            bk.data() + r * 4 * NTT_N, r == 0 ? bk.data() + 8 * NTT_N : nullptr, r, par);
        });
        both(PAIR_THREADS, [&](int r, int tid) { pair_inv3_a(tid, w[r].data(), par); });
        both(PAIR_THREADS, [&](int r, int tid) { pair_inv3_b(tid, w[r].data(), par); });
        both(PAIR_INV_WORKERS, [&](int r, int tid) { pair_inv2(tid, w[r].data(), par); });
        both(PAIR_THREADS, [&](int r, int tid) { pair_inv1_a(tid, w[r].data(), T.inv.data(), par); });
        both(PAIR_THREADS, [&](int r, int tid) { pair_inv1_b(tid, acc[r], w[r].data(), par); });
    }
}

extern "C" {

// the pair shape: `steps` CMux steps with rotation amounts rots[0 .. steps), all with the same key row
void emul_phase_steps_pair(i32 *acc_io, const u64 *bk_ref_row, const int *rots, int steps)
{
    pair_steps(acc_io, bk_ref_row, rots, steps);
}

void emul_phase_step(i32 *acc_io, const u64 *bk_ref_row, const int *rot, int nct)
{
    phase_step<BrDefault>(acc_io, bk_ref_row, rot, nct);
}
// the wide shape (one ciphertext on 256 threads)
void emul_phase_step_wide(i32 *acc_io, const u64 *bk_ref_row, const int *rot)
{
    phase_step<BrWide>(acc_io, bk_ref_row, rot, 1);
}
// the wide2 shape (one ciphertext on 512 threads: split forward and inverse phases)
void emul_phase_step_wide2(i32 *acc_io, const u64 *bk_ref_row, const int *rot)
{
    phase_step<BrWide2>(acc_io, bk_ref_row, rot, 1);
}

void emul_ff_shl_var(const u64 *in, const int *s, u64 *out, size_t n)
{ for (size_t i = 0; i < n; i++) out[i] = ff_shl_var(in[i], s[i]); }
void emul_ff_mul(const u64 *a, const u64 *b, u64 *out, size_t n)
{ for (size_t i = 0; i < n; i++) out[i] = ff_mul(a[i], b[i]); }
void emul_ff_add(const u64 *a, const u64 *b, u64 *out, size_t n)
{ for (size_t i = 0; i < n; i++) out[i] = ff_add(a[i], b[i]); }
void emul_ff_sub(const u64 *a, const u64 *b, u64 *out, size_t n)
{ for (size_t i = 0; i < n; i++) out[i] = ff_sub(a[i], b[i]); }

}  // extern "C"

// ---- the FFT external product (br_fft.cuh) ----------------------------------------------------------------------
// the two limb spectra of every key polynomial of `rows` reference rows (2,2,2,1024 Montgomery NTT values each), in the
// layout the kernels read: rows x [m][limb][512] complex = rows x FFT_ROW_U64 doubles' bits (kernels.cuh:
// fft_key_kernel computes the same on the device)
static void fft_key_row(const u64 *bk_ref_row, const FftTables &T, cplx *out)
{
    std::vector<u64> plain(NTT_N);
    std::vector<i32> k(NTT_N);
    std::vector<cplx> f(FFT_STRIDE);
    for (int m = 0; m < 8; m++) {
        for (int x = 0; x < NTT_N; x++) plain[x] = ff_mul(ff_canon(bk_ref_row[m * NTT_N + x]), FF_RINV);
        emul_ntt_inverse_i32(plain.data(), k.data(), 1);
        for (int limb = 0; limb < 2; limb++) {
            for (int t = 0; t < 64; t++) fft_key_phase1(t, k.data(), limb, f.data(), T);
            for (int t = 0; t < 64; t++) fft_fwd2(t, f.data(), T);
            for (int t = 0; t < 64; t++) fft_key_phase3_store(t, f.data(), out + (m * 2 + limb) * FFT_M);
        }
    }
}

static const FftTables &fft_tables()
{
    static FftTables T;
    static bool init = false;
    if (!init) { make_fft_tables(T); init = true; }
    return T;
}

extern "C" {

// the twiddle tables of the FFT kernel: tw (FFT_M complex) then tw2 (64 complex) as interleaved doubles, and the pass-1
// constants cos(pi j / 16), j = 0..8
void emul_fft_tables(double *tw, double *cos16)
{
    memcpy(tw, &fft_tables(), sizeof(FftTables));
    for (int j = 0; j <= 8; j++) cos16[j] = fft_cos16(j);
}

void emul_fft_key_spectra(const u64 *bk_ref, u64 *out, size_t rows)
{
    for (size_t r = 0; r < rows; r++)
        fft_key_row(bk_ref + r * 8 * NTT_N, fft_tables(), reinterpret_cast<cplx *>(out + r * FFT_ROW_U64));
}

// One CMux step (rot != NULL) or plain external product (rot == NULL: acc <- key (x) acc) of the FFT kernel for `nct`
// ciphertexts (acc: nct x 2 x 1024), phase by phase as the kernel runs them.  *err_max: the largest distance to the
// nearest integer seen before rounding, over all output coefficients.
void emul_fft_step(i32 *acc, const u64 *bk_ref_row, const int *rot, int nct, double *err_max)
{
    const FftTables &T = fft_tables();
    std::vector<cplx> key(FFT_KEY_SPECTRA * FFT_M);
    fft_key_row(bk_ref_row, T, key.data());
    std::vector<cplx> w((size_t)nct * 4 * FFT_STRIDE);
    *err_max = 0;
    for (int c = 0; c < nct; c++)
        for (int mi = 0; mi < 2; mi++)
            for (int t = 0; t < 64; t++) {
                cplx *f2 = w.data() + (c * 4 + mi * 2) * FFT_STRIDE;
                if (rot) fft_step_fwd1<true>(t, acc + (c * 2 + mi) * NTT_N, f2, T, rot[c]);
                else fft_step_fwd1<false>(t, acc + (c * 2 + mi) * NTT_N, f2, T, 0);
            }
    for (int s = 0; s < nct * 4; s++) for (int t = 0; t < 64; t++) fft_fwd2(t, w.data() + s * FFT_STRIDE, T);
    for (int s = 0; s < nct * 4; s++) for (int t = 0; t < 64; t++) fft_fwd3(t, w.data() + s * FFT_STRIDE);
    for (int i = 0; i < FFT_M; i++) fft_step_mac(i, w.data(), 4 * FFT_STRIDE, nct, key.data());
    for (int s = 0; s < nct * 4; s++) for (int t = 0; t < 64; t++) fft_inv3(t, w.data() + s * FFT_STRIDE, T);
    for (int s = 0; s < nct * 4; s++) for (int t = 0; t < 64; t++) fft_inv2(t, w.data() + s * FFT_STRIDE);
    for (int c = 0; c < nct; c++)
        for (int mo = 0; mo < 2; mo++)
            for (int t = 0; t < 64; t++) {
                const cplx *f2 = w.data() + (c * 4 + mo * 2) * FFT_STRIDE;
                if (rot) fft_step_inv1<true>(t, acc + (c * 2 + mo) * NTT_N, f2, T, err_max);
                else fft_step_inv1<false>(t, acc + (c * 2 + mo) * NTT_N, f2, T, err_max);
            }
}

}  // extern "C"
