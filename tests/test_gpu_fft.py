"""GPU tests of the FP64 FFT throughput kernel (csrc/fft_kernels.cuh): the key spectra nb_bk_prepare computes on the
device equal the host emulator's bit for bit, and gate_nand / gate_mux give the same bits through the FFT kernel and the
NTT kernel (NUFHE_B200_FFT=1 / 0), and the oracle's, at batches below and above the shape boundaries."""
import ctypes
import os

import numpy
import pytest

import gen_inputs as G
from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def keys():
    return O.OracleKeys(G.GATE_SEED)


def _engine(monkeypatch, fft, small_shapes_off):
    from nufhe_b200.engine import Engine
    monkeypatch.setenv('NUFHE_B200_FFT', '1' if fft else '0')
    if small_shapes_off:       # the throughput shape below wide_max, as in test_all_cta_shapes_give_the_same_bits
        for k in ('NUFHE_B200_WIDE_MAX', 'NUFHE_B200_WIDE2_MAX', 'NUFHE_B200_PAIR_MAX'):
            monkeypatch.setenv(k, '0')
    else:
        for k in ('NUFHE_B200_WIDE_MAX', 'NUFHE_B200_WIDE2_MAX', 'NUFHE_B200_PAIR_MAX'):
            monkeypatch.delenv(k, raising=False)
    return Engine()


def test_fft_key_spectra_equal_the_host_emulator(keys, monkeypatch):
    eng = _engine(monkeypatch, True, False)
    rows = 3
    bk = numpy.ascontiguousarray(keys.bk[:rows])
    bk_int = eng.to_host(eng.bk_prepare(eng.to_device(bk)), True).reshape(-1)
    row_u64 = eng.lib.nb_bk_row_u64()
    ntt_u64 = 10 * 1024
    spectra = bk_int[rows * ntt_u64:rows * row_u64]
    emul = ctypes.CDLL(os.path.join(ROOT, 'nufhe_b200', 'csrc', 'libnb_host_emul.so'))
    want = numpy.empty(rows * (row_u64 - ntt_u64), numpy.uint64)
    emul.emul_fft_key_spectra(bk.ctypes.data_as(ctypes.c_void_p), want.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(rows))
    assert (spectra.view(numpy.uint64) == want).all()


def _nand(eng, dk, a, b):
    bk_int, ks = dk
    num, den, sa, sb = O.GATE_TABLE['nand']
    da = (eng.to_device(a[0]), eng.to_device(a[1]))
    db = (eng.to_device(b[0]), eng.to_device(b[1]))
    ext = eng.bootstrap_extract(da, db, O.phase_to_t32(num, den), sa, sb, O.MU, bk_int)
    ra, rb, _ = eng.keyswitch(ks, ext)
    return eng.to_host(ext[0]), eng.to_host(ext[1]), eng.to_host(ra), eng.to_host(rb)


def _mux(eng, dk, a, b, c):
    bk_int, ks = dk
    d = [(eng.to_device(x[0]), eng.to_device(x[1])) for x in (a, b, c)]
    and_const = O.phase_to_t32(-1, 8)
    u1, u2 = eng.bootstrap_extract2((d[0], d[1], and_const, 1, 1), (d[0], d[2], and_const, -1, 1), O.MU, bk_int)
    ma, mb, _ = eng.keyswitch(ks, u1, u2, c=O.phase_to_t32(1, 8))
    return eng.to_host(u1[0]), eng.to_host(u2[0]), eng.to_host(ma), eng.to_host(mb)


def _sub(x, rows):
    return (numpy.ascontiguousarray(x[0][rows]), numpy.ascontiguousarray(x[1][rows]))


@pytest.mark.parametrize('batch', [301, 592, 700, 4096, 65536])
@pytest.mark.parametrize('gate', ['nand', 'mux'])
def test_fft_and_ntt_kernels_give_the_same_bits(keys, monkeypatch, gate, batch):
    if gate == 'mux' and batch == 65536:
        pytest.skip('two bootstraps of 65536 ciphertexts: covered by nand at this size')
    rng = G.rs(5000 + batch)
    nin = 3 if gate == 'mux' else 2
    bits = rng.randint(0, 2, (nin, batch)).astype(bool)
    cts = [keys.encrypt(b) for b in bits]
    small = batch < 1000          # below wide_max on a B200: force the throughput shape
    outs = []
    for fft in (True, False):
        eng = _engine(monkeypatch, fft, small)
        dk = (eng.bk_prepare(eng.to_device(keys.bk)), (eng.to_device(keys.ks_a), eng.to_device(keys.ks_b),
                                                       eng.to_device(keys.ks_cv)))
        outs.append(_nand(eng, dk, *cts) if gate == 'nand' else _mux(eng, dk, *cts))
        del eng, dk
    for x, y in zip(*outs):
        assert (x == y).all()
    # the oracle on a strided subset (every ciphertext of the FFT run is checked against the NTT run above)
    rows = numpy.arange(0, batch, max(1, batch // 6))[:6]
    sub = [_sub(c, rows) for c in cts]
    if gate == 'nand':
        want = O.gate_binary('nand', sub[0], sub[1], keys.bk, keys.ks)
        got = (outs[0][2][rows], outs[0][3][rows])
        assert (keys.decrypt(got) == ~(bits[0][rows] & bits[1][rows])).all()
    else:
        want = O.gate_mux(sub[0], sub[1], sub[2], keys.bk, keys.ks)
        got = (outs[0][2][rows], outs[0][3][rows])
        assert (keys.decrypt(got) == numpy.where(bits[0][rows], bits[1][rows], bits[2][rows])).all()
    assert (got[0] == want[0]).all() and (got[1] == want[1]).all()
