"""CPU-only tests: host logic of the nufhe-compatible API, the C ABI surface, and the host emulation
of the per-lane GPU transform code against the oracle."""
import ctypes
import os
import re

import numpy
import pytest

import gen_inputs as G
from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_capi_library_loads_and_exports_every_declared_symbol():
    from nufhe_b200 import _native
    lib = _native.load()
    hdr = open(os.path.join(ROOT, 'include', 'nufhe_b200.h')).read()
    declared = set(re.findall(r'\b(nb_[a-z0-9_]+)\s*\(', hdr)) - {'nb_ctx'}
    assert declared == set(_native.SIGNATURES)
    for name in declared:
        assert hasattr(lib, name), name


def test_capi_rejects_null_context_without_gpu():
    from nufhe_b200 import _native
    lib = _native.load()
    assert lib.nb_ctx_synchronize(None) == _native.NB_EINVAL
    assert lib.nb_ntt_forward_i32(None, None, None, 4) == _native.NB_EINVAL


def test_engine_fails_loudly_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip('CUDA present')
    from nufhe_b200.engine import Engine
    with pytest.raises(RuntimeError):
        Engine()
    import nufhe_b200 as nufhe
    with pytest.raises(RuntimeError):
        nufhe.Context()


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, 'nufhe_b200')
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h', '.cpp')):
                src = open(os.path.join(dirpath, f)).read()
                assert 'import oracle' not in src and 'from oracle' not in src, f
                assert 'libnufhe_oracle' not in src, f
                assert 'fake_engine' not in src and 'FakeEngine' not in src, f      # the CPU test double stays in tests/
    for extra in ('bench.py',):
        src = open(os.path.join(ROOT, extra)).read()
        assert 'fake_engine' not in src and 'FakeEngine' not in src, extra


def test_parameters_and_shapes():
    import nufhe_b200 as nufhe
    from nufhe_b200.gates import result_shape, check_shape
    p = nufhe.NuFHEParameters()
    assert p == nufhe.NuFHEParameters() and hash(p) == hash(nufhe.NuFHEParameters())
    assert p.in_out_params.size == 500 and p.tgsw_params.tlwe_params.polynomial_degree == 1024
    assert int(p.tgsw_params.offset) == -2145386496            # SURVEY.md section 8 a8
    assert p.ks_decomp_length == 8 and p.ks_log2_base == 2
    with pytest.raises(ValueError):
        nufhe.NuFHEParameters(transform_type='FFT')
    with pytest.raises(AssertionError):
        nufhe.NuFHEParameters(transform_type='DCT')
    # mask size 2 exists on the multi-kernel path only, like in the reference (blind_rotate.py:53-58, performance.py:183-185)
    p2 = nufhe.NuFHEParameters(tlwe_mask_size=2)
    assert p2 != p and p2.tgsw_params.tlwe_params.extracted_lweparams.size == 2048

    class Dev:
        pass
    assert nufhe.PerformanceParameters(p).for_device(Dev()).single_kernel_bootstrap
    assert not nufhe.PerformanceParameters(p2).for_device(Dev()).single_kernel_bootstrap
    assert not nufhe.PerformanceParameters(p, single_kernel_bootstrap=False).for_device(Dev()).single_kernel_bootstrap
    with pytest.raises(ValueError):
        nufhe.PerformanceParameters(p2, single_kernel_bootstrap=True).for_device(Dev())
    pp = nufhe.PerformanceParameters(p, single_kernel_bootstrap=True)
    assert pp == nufhe.PerformanceParameters(p, single_kernel_bootstrap=True)
    assert pp != nufhe.PerformanceParameters(p)
    with pytest.raises(AssertionError):
        nufhe.PerformanceParameters(p, ntt_base_method='fortran')
    # broadcasting rules of gates.py:51-78
    assert result_shape((3, 1), (4,)) == (3, 4)
    assert result_shape((2, 3), (1, 3), (3,)) == (2, 3)
    with pytest.raises(ValueError):
        result_shape((2, 3), (4, 3))

    class S:
        def __init__(self, shape):
            self.shape = shape
    check_shape(S((5, 2, 3)), S((2, 3)), S((3,)))
    with pytest.raises(ValueError):
        check_shape(S((2, 3)), S((5, 2, 3)))
    with pytest.raises(ValueError):
        check_shape(S((2, 4)), S((2, 3)))
    with pytest.raises(ValueError):                   # the derived shape must EQUAL the trailing dims (gates.py:73)
        check_shape(S((3, 4)), S((1, 4)))
    check_shape(S((3, 4)), S((4,)))
    check_shape(S((3, 4)), S(()))                     # a scalar (gate_constant with one bit)
    assert result_shape((1, 4)) == (1, 4) and result_shape((7,), (1,)) == (7,)


def test_encodings():
    from nufhe_b200.numeric_functions import phase_to_t32, double_to_t32
    from nufhe_b200.api_low_level import bool_to_t32, t32_to_bool
    assert int(phase_to_t32(1, 8)) == 2**29 and int(phase_to_t32(-1, 8)) == -2**29
    assert int(phase_to_t32(1, 4)) == 2**30 and int(phase_to_t32(-1, 4)) == -2**30
    assert (bool_to_t32([True, False]) == [2**29, -2**29]).all()
    assert (t32_to_bool(numpy.array([5, -5, 0])) == [True, False, False]).all()
    assert (double_to_t32(numpy.array([0.25, -0.25, 1.25])) == [2**30, -2**30, 2**30]).all()


def test_rng_matches_reference_semantics():
    import nufhe_b200 as nufhe
    r1, r2 = nufhe.DeterministicRNG(5), numpy.random.RandomState(5)
    assert (r1.uniform_bool((7,)) == r2.randint(0, 2, size=(7,), dtype=numpy.int32)).all()
    assert (r1.uniform_torus32((3, 2)) == r2.randint(-2**31, 2**31, size=(3, 2), dtype=numpy.int32)).all()
    assert (r1.gauss((4,), 0.5) == r2.normal(size=(4,), scale=0.5)).all()
    s = nufhe.SecureRNG()
    assert s.uniform_bool((3, 5)).shape == (3, 5) and set(numpy.unique(s.uniform_bool((64,)))) <= {0, 1}
    assert s.uniform_torus32((9,)).dtype == numpy.int32
    g = s.gauss((1001,), 2.0)
    assert g.shape == (1001,) and 1.0 < g.std() < 3.0


def test_secure_rng_statistics():
    """SecureRNG is our own sampler (no seed, nothing to match byte for byte): check the distributions instead.
    Bounds are ~6 sigma of the estimator, so a correct sampler fails with probability < 1e-8."""
    from scipy import stats
    import nufhe_b200 as nufhe
    s = nufhe.SecureRNG()
    n = 400000
    bits = s.uniform_bool((n,))
    assert bits.dtype == numpy.int32 and abs(bits.mean() - 0.5) < 6 * 0.5 / n**0.5
    t = s.uniform_torus32((n,)).astype(numpy.float64) / 2**32
    assert abs(t.mean()) < 6 * (1 / 12**0.5) / n**0.5 and abs(t.var() - 1 / 12) < 0.002
    assert stats.kstest(t + 0.5, 'uniform').pvalue > 1e-6
    u = s._open_unit_interval(n)
    assert u.min() > 0.0 and u.max() < 1.0                     # open interval: log(u) is always finite
    sigma = 1 / 2**15 * (2 / numpy.pi)**0.5                    # the scheme's LWE noise, api_low_level.py:58-59
    g = s.gauss((n + 1,), sigma)                               # odd count: the last pair is cut
    assert g.shape == (n + 1,) and numpy.isfinite(g).all()
    assert abs(g.mean()) < 6 * sigma / n**0.5 and abs(g.std() / sigma - 1) < 6 / (2 * n)**0.5
    assert stats.kstest(g / sigma, 'norm').pvalue > 1e-6
    assert abs(stats.kurtosis(g)) < 0.05 and abs(stats.skew(g)) < 0.03
    assert s.gauss((2, 3, 5), 1.0).shape == (2, 3, 5)
    # the two halves of the polar pairs are uncorrelated
    assert abs(numpy.corrcoef(g[:n // 2], g[n // 2:n])[0, 1]) < 6 / (n // 2)**0.5


# ---- the per-lane GPU transform code, executed on the host (csrc/host_emul.cpp) ------------------

@pytest.fixture(scope='module')
def emul():
    path = os.path.join(ROOT, 'nufhe_b200', 'csrc', 'libnb_host_emul.so')
    if not os.path.exists(path):
        import __graft_entry__ as g
        g.build()
    return ctypes.CDLL(path)


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def test_lane_ntt_matches_oracle(emul):
    rng = G.rs(5)
    x = G.ff_numbers(rng, (3, 1024))
    out = numpy.empty_like(x)
    emul.emul_ntt_forward(_p(x), _p(out), ctypes.c_size_t(3))
    assert (out == O.ntt_forward_u64(x)).all()
    emul.emul_ntt_inverse(_p(x), _p(out), ctypes.c_size_t(3))
    assert (out == O.ntt_inverse_u64(x)).all()


def test_lane_ntt_matches_reference_golden(emul, golden):
    g = golden('ntt')
    _, x_u64 = G.ntt_inputs()
    out = numpy.empty_like(x_u64)
    emul.emul_ntt_forward(_p(x_u64), _p(out), ctypes.c_size_t(x_u64.shape[0]))
    assert (out == g['fwd_u64']).all()
    emul.emul_ntt_inverse(_p(x_u64), _p(out), ctypes.c_size_t(x_u64.shape[0]))
    assert (out == g['inv_u64']).all()


def test_lane_ntt_i32_conversion(emul, golden):
    """The stand-alone transforms with Torus32 on the natural-order side: the forward pass fuses the conversion with
    the twist (ff_twist_i32), the inverse negates after the conversion.  Edge coefficients (0, +-1, +-2^31) and
    random ones against the reference's goldens and the oracle."""
    g = golden('ntt')
    x_i32, x_u64 = G.ntt_inputs()
    out = numpy.empty(x_i32.shape, numpy.uint64)
    emul.emul_ntt_forward_i32(_p(x_i32), _p(out), ctypes.c_size_t(x_i32.shape[0]))
    assert (out == g['fwd_i32']).all()
    back = numpy.empty(x_u64.shape, numpy.int32)
    emul.emul_ntt_inverse_i32(_p(x_u64), _p(back), ctypes.c_size_t(x_u64.shape[0]))
    assert (back == g['inv_i32']).all()
    rng = G.rs(9)
    x = G.torus32(rng, (4, 1024))
    x[0, :8] = [0, 1, -1, 2**31 - 1, -2**31, -2**31 + 1, 2**30, -2**30]
    x[1, :] = -2**31
    x[2, :] = 2**31 - 1
    out = numpy.empty(x.shape, numpy.uint64)
    emul.emul_ntt_forward_i32(_p(x), _p(out), ctypes.c_size_t(4))
    assert (out == O.ntt_forward_i32(x)).all()
    back = numpy.empty(x.shape, numpy.int32)
    emul.emul_ntt_inverse_i32(_p(out), _p(back), ctypes.c_size_t(4))
    assert (back == x).all()
    y = G.ff_numbers(rng, (3, 1024))
    back = numpy.empty(y.shape, numpy.int32)
    emul.emul_ntt_inverse_i32(_p(y), _p(back), ctypes.c_size_t(3))
    assert (back == O.ntt_inverse_i32(y)).all()


def test_lane_field_ops_match_oracle(emul, golden):
    g = golden('arithmetic')
    a, b, s = G.arithmetic_inputs()
    a, b = a % numpy.uint64(G.P), b % numpy.uint64(G.P)
    out = numpy.empty_like(a)
    n = ctypes.c_size_t(a.size)
    emul.emul_ff_mul(_p(a), _p(b), _p(out), n)
    assert (out == g['mul']).all()
    emul.emul_ff_add(_p(a), _p(b), _p(out), n)
    assert (out == g['add']).all()
    emul.emul_ff_sub(_p(a), _p(b), _p(out), n)
    assert (out == g['sub']).all()
    si = s.astype(numpy.int32)
    emul.emul_ff_shl_var(_p(a), _p(si), _p(out), n)
    assert (out == g['lsh']).all()


def test_phase_structured_step_matches_oracle(emul):
    """csrc/br_phases.cuh (the fused bootstrap's CTA-wide phases) executed on the host: plain external
    product and one rotate-and-accumulate CMux step, random field key, edge rotation amounts."""
    rng = G.rs(77)
    bk = G.ff_numbers(rng, (2, 2, 2, 2, 1024))
    for nct in range(1, emul.emul_phase_ct() + 1):
        acc = G.torus32(rng, (nct, 2, 1024))
        a = acc.copy()
        emul.emul_phase_step(_p(a), _p(bk[1]), None, ctypes.c_int(nct))
        assert (a == O.tgsw_external_mul(acc, bk, 1)).all()
        rot = numpy.array([0, 1024, 1023, 2047][:nct], numpy.int32)
        a = acc.copy()
        emul.emul_phase_step(_p(a), _p(bk[0]), _p(rot), ctypes.c_int(nct))
        assert (a == O.blind_rotate(acc, bk[0:1], rot.reshape(nct, 1))).all()
    # the wide CTA shapes (one ciphertext on 256 / 512 threads, used for small batches): the inverse phases -- and in
    # the 512-thread shape also the forward phases -- run split, two threads per 16-element task, 8 elements each
    for step in (emul.emul_phase_step_wide, emul.emul_phase_step_wide2):
        for r in (0, 5, 1024, 2047):
            acc = G.torus32(rng, (1, 2, 1024))
            a = acc.copy()
            step(_p(a), _p(bk[1]), None)
            assert (a == O.tgsw_external_mul(acc, bk, 1)).all()
            rot = numpy.array([r], numpy.int32)
            a = acc.copy()
            step(_p(a), _p(bk[0]), _p(rot))
            assert (a == O.blind_rotate(acc, bk[0:1], rot.reshape(1, 1))).all()


def test_pair_shape_steps_match_oracle(emul):
    """The pair shape (one ciphertext on a cluster of two CTAs, csrc/br_phases.cuh) on the host: two emulated CTAs,
    the partial sums of the MAC exchanged through each other's work polynomials.  Several consecutive steps cover both
    parities of the exchange area and whatever one step leaves behind in shared memory for the next."""
    rng = G.rs(78)
    bk = G.ff_numbers(rng, (2, 2, 2, 2, 1024))
    for rots in ([0], [1024], [5, 2047, 1023, 1], [2047, 0, 77]):
        acc = G.torus32(rng, (1, 2, 1024))
        a = acc.copy()
        r = numpy.array(rots, numpy.int32)
        emul.emul_phase_steps_pair(_p(a), _p(bk[0]), _p(r), ctypes.c_int(len(rots)))
        rows = numpy.stack([bk[0]] * len(rots))
        assert (a == O.blind_rotate(acc, rows, r.reshape(1, -1))).all()


def test_committed_traffic_capture_belongs_to_the_built_kernel():
    """bench.py quotes `roofline.traffic` from profiles/r2_traffic.json only when the kernel of the running library has
    the same static per-phase instruction counts as the one the ncu capture was taken on (tools/sass_stats.py, no GPU
    needed).  Guard against kernel edits that forget to re-capture: the committed fingerprint must match this build."""
    import json
    import shutil
    import subprocess
    import sys
    if not (shutil.which('cuobjdump') and shutil.which('nvdisasm')):
        pytest.skip('CUDA binary utilities not on PATH')
    with open(os.path.join(ROOT, 'profiles', 'r2_traffic.json')) as f:
        fp = json.load(f)['kernel_fingerprint']
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tools', 'sass_stats.py'), '--json'], capture_output=True,
                       text=True, timeout=300)
    cur = json.loads(r.stdout)
    assert cur['phases'] == fp['phases'] and cur['per_thread_step_total'] == fp['per_thread_step_total']
    assert cur['per_thread_step_total'] > 5000          # the tool found the step loop


def test_uint_bit_helpers_roundtrip():
    from nufhe_b200.operators_integer import uintarray_to_bitarray, bitarray_to_uintarray
    xs = numpy.array([[0, 1, 255], [128, 77, 200]], numpy.uint8)
    bits = uintarray_to_bitarray(xs)
    assert bits.shape == (2, 3, 8) and bits[0, 1].tolist() == [False] * 7 + [True]
    assert (bitarray_to_uintarray(bits) == xs).all()
    ys = numpy.array([0, 1, 2**31, 2**32 - 1], numpy.uint32)
    assert (bitarray_to_uintarray(uintarray_to_bitarray(ys)) == ys).all()


def test_bench_dump_outputs_exact_and_bounded(tmp_path):
    """bench.py --dump-outputs: every int32 survives the float64 file exactly; above the size limit a seeded sample
    of whole ciphertexts is written, the same one every time, and the files stay within the limit."""
    import bench
    rng = numpy.random.RandomState(3)

    def case(n):
        return (rng.randint(-2**31, 2**31, (n, 500), dtype=numpy.int32), rng.randint(-2**31, 2**31, n, dtype=numpy.int32),
                rng.uniform(0, 1e-3, n).astype(numpy.float32))

    a, b, cv = case(64)
    bench.dump_outputs(str(tmp_path / 'small'), a, b, cv)
    got = {k: numpy.load(str(tmp_path / 'small' / (k + '.npy'))) for k in ('a', 'b', 'current_variances')}
    assert got['a'].dtype == numpy.float64 and (got['a'] == a).all() and (got['b'] == b).all()
    assert got['current_variances'].dtype == numpy.float32 and (got['current_variances'] == cv).all()
    assert not (tmp_path / 'small' / 'rows.npy').exists()

    a, b, cv = case(20000)                      # 20000 x 4020 bytes > 64 MB
    for d in ('big1', 'big2'):
        bench.dump_outputs(str(tmp_path / d), a, b, cv)
    assert sum(f.stat().st_size for f in (tmp_path / 'big1').iterdir()) <= bench.DUMP_LIMIT_BYTES
    rows = numpy.load(str(tmp_path / 'big1' / 'rows.npy')).astype(numpy.int64)
    assert (numpy.diff(rows) > 0).all() and len(rows) > 15000
    assert (rows == numpy.load(str(tmp_path / 'big2' / 'rows.npy'))).all()
    assert (numpy.load(str(tmp_path / 'big1' / 'a.npy')) == a[rows]).all()
    assert (numpy.load(str(tmp_path / 'big1' / 'b.npy')) == b[rows]).all()


def test_pickle_wire_compatibility_with_reference_parameter_classes():
    """The parameter objects nufhe pickles into every dump: ours carry the same attributes and, with
    compat.use_reference_pickle_paths(), the same class paths; a pickle made by the REFERENCE's classes
    (committed as tests/golden/ref_params.pkl by make_golden.py) loads into ours and compares equal."""
    import pickle
    import subprocess
    import sys
    code = r'''
import pickle, sys
sys.path.insert(0, %r)
import nufhe_b200
from nufhe_b200 import compat
compat.use_reference_pickle_paths()
p = nufhe_b200.NuFHEParameters()
blob = pickle.dumps(p)
assert b'nufhe.api_low_level' in blob and b'nufhe_b200' not in blob, blob[:200]
q = pickle.loads(blob)
assert q == p and q.in_out_params == p.in_out_params and q.tgsw_params == p.tgsw_params
ref = pickle.load(open(%r, 'rb'))
assert type(ref).__name__ == 'NuFHEParameters' and type(ref).__module__ == 'nufhe.api_low_level'
assert ref == p
assert ref.in_out_params.size == 500 and ref.tgsw_params.tlwe_params.polynomial_degree == 1024
assert int(ref.tgsw_params.offset) == int(p.tgsw_params.offset)
assert (ref.tgsw_params.base_powers == p.tgsw_params.base_powers).all()
print('ok')
''' % (ROOT, os.path.join(ROOT, 'tests', 'golden', 'ref_params.pkl'))
    out = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True)
    assert out.returncode == 0 and 'ok' in out.stdout, out.stderr
