// tables.h -- host-side construction of the constant tables the kernels consume:
//   * the middle twiddles psi^(j2 (2 k1 + 1)) of the transform passes (br_phases.cuh), forward and inverse;
//   * 512 * NTT(all-ones), used for the correction planes of the engine-format bootstrap key.
// Host only (uses unsigned __int128); shared by the CUDA library and the host lane emulator.
#pragma once
#include <vector>
#include "ntt_lane.cuh"
#include "br_phases.cuh"
#include "br_fft.cuh"
#include <cmath>

namespace nb {

inline u64 h_mul(u64 a, u64 b) { return (u64)(((unsigned __int128)a * b) % FF_P); }
inline u64 h_pow(u64 a, u64 e) { u64 r = 1; while (e) { if (e & 1) r = h_mul(r, a); a = h_mul(a, a); e >>= 1; } return r; }
inline u64 h_inv(u64 a) { return h_pow(a, FF_P - 2); }

constexpr u64 ROOT_GEN = 0xa70dc47e4cbdf43fULL;          // nufhe/transform/ntt_cpu.py:109

// Tables of the phase-structured bootstrap kernel (br_phases.cuh): [row][j2], 64 entries per row.
struct PhaseTables {
    std::vector<u64> fwd, inv;
    std::vector<u64> ones512;   // 512 * NTT(1,1,...,1)[k] in natural order: 512 * 2 / (1 - psi^(2k+1))
    PhaseTables() : fwd(NTT_N), inv(NTT_N), ones512(NTT_N)
    {
        {
            const u64 psi0 = h_pow(ROOT_GEN, (1ULL << 32) / 2048);
            for (int k = 0; k < NTT_N; k++) {
                u64 r = h_pow(psi0, 2 * k + 1);
                u64 denom = (FF_P + 1 - r) % FF_P;          // 1 - r
                ones512[k] = h_mul(1024, h_inv(denom));     // sum_j r^j = (1 - r^1024) / (1 - r) = 2 / (1 - r)
            }
        }
        const u64 psi = h_pow(ROOT_GEN, (1ULL << 32) / 2048);
        const u64 psi_inv = h_inv(psi), n_inv = h_inv(NTT_N);
        for (int row = 0; row < 16; row++)
            for (int j2 = 0; j2 < 64; j2++) {
                int e = w_twiddle_exponent(row, j2);
                fwd[row * 64 + j2] = h_pow(psi, e);
                inv[row * 64 + j2] = h_mul(h_pow(psi_inv, e), n_inv);
            }
    }
};

// Twiddles of the FFT external product (br_fft.cuh), each component computed in long double and rounded once to
// double: |error| <= 2^-53 per component (the bound in DESIGN.md section 8 uses this).
inline void make_fft_tables(FftTables &T)
{
    const long double pi = 3.141592653589793238462643383279502884L;
    auto w = [&](int m) { m &= FFT_M - 1; return cplx{(double)cosl(2 * pi * m / FFT_M), (double)sinl(2 * pi * m / FFT_M)}; };
    for (int m = 0; m < FFT_M; m++) {                  // omega^(t (1 + 4 k0)), t = m & 63, k0 = m >> 6
        const int e = ((m & 63) * (1 + 4 * (m >> 6))) & (2 * NTT_N - 1);
        T.tw[m] = cplx{(double)cosl(pi * e / NTT_N), (double)sinl(pi * e / NTT_N)};
    }
    for (int m = 0; m < 64; m++) T.tw2[m] = w(8 * (m >> 3) * (m & 7));
}

}  // namespace nb
