"""CPU-only tests of the FFT external product (csrc/br_fft.cuh) executed on the host (csrc/host_emul.cpp): the CMux
step and the plain external product of the FP64 kernel must equal the oracle's exact results bit for bit, also at the
magnitude extremes, with a wide margin between the largest rounding distance and 1/2."""
import ctypes
import os

import numpy
import pytest

import gen_inputs as G
from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def emul():
    path = os.path.join(ROOT, 'nufhe_b200', 'csrc', 'libnb_host_emul.so')
    if not os.path.exists(path):
        import __graft_entry__ as g
        g.build()
    lib = ctypes.CDLL(path)
    lib.emul_fft_step.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                  ctypes.POINTER(ctypes.c_double)]
    return lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _key(raw):
    """(rows, 2, 2, 2, 1024) int32 TGSW polynomials -> the reference's transformed key (NTT, Montgomery form)."""
    raw = numpy.ascontiguousarray(raw, numpy.int32)
    bk = numpy.empty(raw.shape, numpy.uint64)
    O.lib().orc_bk_transform(_p(bk), _p(raw), ctypes.c_size_t(raw.size // 1024))
    return bk


def _step(emul, acc, bk_row, rot):
    a = numpy.ascontiguousarray(acc).copy()
    err = ctypes.c_double()
    emul.emul_fft_step(_p(a), _p(numpy.ascontiguousarray(bk_row)), None if rot is None else _p(rot), a.shape[0],
                       ctypes.byref(err))
    return a, err.value


def test_fft_step_matches_oracle(emul):
    rng = G.rs(91)
    bk = _key(rng.randint(-2**31, 2**31, size=(2, 2, 2, 2, 1024), dtype=numpy.int32))
    for nct in (1, 2, 4):
        acc = G.torus32(rng, (nct, 2, 1024))
        got, err = _step(emul, acc, bk[1], None)
        assert (got == O.tgsw_external_mul(acc, bk, 1)).all()
        assert err < 2.0**-6
        for rots in ([0] * nct, [1023] * nct, [1024] * nct, [2047] * nct, list(rng.randint(0, 2048, nct))):
            rot = numpy.array(rots, numpy.int32)
            got, err = _step(emul, acc, bk[0], rot)
            assert (got == O.blind_rotate(acc, bk[0:1], rot.reshape(nct, 1))).all(), rots
            assert err < 2.0**-6


def test_fft_step_at_the_magnitude_extremes(emul):
    """Every digit -512 (accumulator coefficients 0x7fe00000 give digit 0 at both levels) and key limbs at +-2^15 with
    signs aligned so that coefficient 0 of every limb convolution reaches 4 * 1024 * 512 * 2^15 = 2^36."""
    raw = numpy.empty((1, 2, 2, 2, 1024), numpy.int64)
    raw[...] = 0x80007fff - 2**32          # limbs (2^15 - 1, -2^15)
    raw[..., 0] = 0x7fff8000               # limbs (-2^15, 2^15)
    bk = _key(raw.astype(numpy.int32))
    acc = numpy.full((2, 2, 1024), 0x7fe00000, numpy.int32)
    got, err = _step(emul, acc, bk[0], None)
    assert (got == O.tgsw_external_mul(acc, bk, 0)).all()
    assert err < 2.0**-6
    # the same key under a rotation: (X^a - 1) ACC with ACC = 0 except the coefficients that make the digits extreme
    rot = numpy.array([0, 1024], numpy.int32)
    got, err = _step(emul, acc, bk[0], rot)
    assert (got == O.blind_rotate(acc, bk, rot.reshape(2, 1))).all()
    assert err < 2.0**-6
