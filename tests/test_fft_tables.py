"""CPU-only tests of the constants of the FFT external product (csrc/br_fft.cuh, built into the host emulator): the
merged pass-1 twiddles and the e^(i pi j / 16) constants are the exact values rounded once, and the key spectra the
merged forward transform computes are the DFT of the folded, twisted key limbs."""
import ctypes
import os

import numpy
import pytest

import gen_inputs as G
from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M = 512
PI = numpy.longdouble('3.14159265358979323846264338327950288')


@pytest.fixture(scope='module')
def emul():
    path = os.path.join(ROOT, 'nufhe_b200', 'csrc', 'libnb_host_emul.so')
    if not os.path.exists(path):
        import __graft_entry__ as g
        g.build()
    lib = ctypes.CDLL(path)
    lib.emul_fft_tables.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    lib.emul_fft_key_spectra.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t]
    return lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _tables(emul):
    tw = numpy.empty((M + 64) * 2, numpy.float64)
    c16 = numpy.empty(9, numpy.float64)
    emul.emul_fft_tables(_p(tw), _p(c16))
    tw = tw[0::2] + 1j * tw[1::2]
    return tw[:M], tw[M:], c16


def test_pass1_twiddles_are_rounded_once(emul):
    """tw[64 k0 + t] = omega^(t (1 + 4 k0)), omega = e^(i pi / 1024), within 2^-53 per component of a long-double
    reference (the per-element bound DESIGN.md section 8 uses); tw2 likewise."""
    tw, tw2, _ = _tables(emul)
    m = numpy.arange(M)
    e = ((m & 63) * (1 + 4 * (m >> 6))) % 2048
    ang = PI * e.astype(numpy.longdouble) / 1024
    assert numpy.abs(tw.real - numpy.cos(ang)).max() <= 2.0**-53
    assert numpy.abs(tw.imag - numpy.sin(ang)).max() <= 2.0**-53
    a = numpy.arange(64)
    ang2 = 2 * PI * (8 * (a >> 3) * (a & 7)).astype(numpy.longdouble) / 512
    assert numpy.abs(tw2.real - numpy.cos(ang2)).max() <= 2.0**-53
    assert numpy.abs(tw2.imag - numpy.sin(ang2)).max() <= 2.0**-53


def test_pass1_constants_are_rounded_once(emul):
    """cos(pi j / 16), j = 0..8 (the sines are cos(pi (8 - j) / 16)): each the double nearest to the exact value."""
    _, _, c16 = _tables(emul)
    ref = numpy.cos(PI * numpy.arange(9, dtype=numpy.longdouble) / 16)
    ref[8] = 0
    assert (c16 == ref.astype(numpy.float64)).all()


def test_key_spectra_are_the_dft_of_the_twisted_limbs(emul):
    rng = G.rs(17)
    raw = rng.randint(-2**31, 2**31, size=(1, 2, 2, 2, 1024), dtype=numpy.int64).astype(numpy.int32)
    bk = numpy.empty(raw.shape, numpy.uint64)
    O.lib().orc_bk_transform(_p(bk), _p(raw), ctypes.c_size_t(raw.size // 1024))
    out = numpy.empty(16 * M * 2, numpy.float64)
    emul.emul_fft_key_spectra(_p(bk), _p(out), ctypes.c_size_t(1))
    got = (out[0::2] + 1j * out[1::2]).reshape(8, 2, M)
    k = numpy.arange(M)
    stored = 64 * (k % 8) + 8 * ((k // 8) % 8) + k // 64        # X[k0 + 8 k1 + 64 k2] sits at 64 k0 + 8 k1 + k2
    omega = numpy.exp(1j * numpy.pi * numpy.arange(M) / 1024)
    polys = raw.reshape(8, 1024).astype(numpy.int64)
    lo = ((polys + 2**15) % 2**16) - 2**15
    hi = (polys - lo) >> 16
    for m in range(8):
        for limb, c in enumerate((lo[m], hi[m])):
            z = (c[:M] + 1j * c[M:]) * omega
            want = numpy.fft.ifft(z)                               # kernel e^(+2 pi i jk / 512), scaled by 1/512
            g = got[m, limb, stored]
            assert numpy.abs(g - want).max() <= 2.0**-30 * numpy.abs(want).max(), (m, limb)
