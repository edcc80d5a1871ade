"""bfReduce parity -- mirrors the sweep of the reference's test/test_reduce.py
(shapes, axes, factors, ops, dtypes, sliced inputs) against the numpy oracle,
plus float-valued data where summation order is visible, plus min/max/stderr
which the reference leaves untested (test/test_reduce.py:114)."""
import numpy as np
import pytest

import bifrost_b200 as bf
from oracle import ops as oracle

pytestmark = pytest.mark.gpu
NP_DT = {'f32': np.float32, 'i16': np.int16, 'i8': np.int8, 'u8': np.uint8, 'u16': np.uint16}


def int_valued(rng, shape, dtype):
    a = ((rng.random(size=shape) * 2 - 1) * 127).astype(np.int8)
    if dtype in ('u8', 'u16'):
        a = np.abs(a)
    return a.astype(NP_DT[dtype])


def run(a, n, axis, op, out_dtype='f32'):
    oshape = list(a.shape)
    oshape[axis] = 1 if n is None else a.shape[axis] // n
    d_a = bf.asarray(a, space='cuda')
    d_b = bf.empty(oshape, dtype=out_dtype, space='cuda')
    bf.reduce(d_a, d_b, op)
    return np.asarray(d_b.copy('system'))


@pytest.mark.parametrize("shape", [(3, 6, 5), (20, 20, 40), (20, 40, 60), (40, 100, 200),
                                   (16, 32, 64), (16, 64, 256), (256, 64, 16)])
def test_real_sweep(shape):
    rng = np.random.default_rng(1234)
    factors = [2, 4, 5, 8, 10, 16, None]
    for axis in range(3):
        for n in factors:
            if n is not None and shape[axis] % n:
                continue
            for op in ['sum', 'mean', 'pwrsum', 'pwrmean', 'min', 'max', 'stderr', 'pwrmin',
                       'pwrmax', 'pwrstderr']:
                for dtype in ['f32', 'i16', 'i8', 'u8']:
                    a = int_valued(rng, shape, dtype)
                    got = run(a, n, axis, op)
                    want = oracle.reduce(a, n, axis, op)
                    np.testing.assert_allclose(got, want, rtol=1e-7, err_msg=str((shape, axis, n, op, dtype)))


@pytest.mark.parametrize("shape", [(20, 20, 40), (16, 64, 256)])
def test_sliced_inputs(shape):
    """test/test_reduce.py:83-109: offset, non-contiguous device views."""
    rng = np.random.default_rng(99)
    for axis in range(3):
        for n in [2, 4, 5, 8]:
            for dtype in ['f32', 'i8', 'i16']:
                a = int_valued(rng, shape, dtype)
                stop = ((a.shape[axis] - 1) // n - 1) * n + 1
                if stop <= 1:
                    continue
                sl = [slice(None)] * 3
                sl[axis] = slice(1, stop)
                sl = tuple(sl)
                d_a = bf.asarray(a, space='cuda')
                view = d_a[sl]
                want = oracle.reduce(a[sl], n, axis, 'sum')
                d_b = bf.empty(want.shape, dtype='f32', space='cuda')
                bf.reduce(view, d_b, 'sum')
                np.testing.assert_allclose(np.asarray(d_b.copy('system')), want, rtol=1e-7)


def test_float_data_keeps_reference_summation_order():
    """With non-integer data the left-to-right fp32 order is observable."""
    rng = np.random.default_rng(5)
    for shape, axis, n in [((64, 4096), 1, 4), ((64, 4096), 1, 16), ((64, 4096), 1, 64),
                           ((4096, 64), 0, 8), ((32, 100, 24), 1, 25), ((7, 33, 1000), 2, None)]:
        a = (rng.normal(size=shape) * 1000).astype(np.float32)
        for op in ['sum', 'mean', 'pwrsum', 'max', 'stderr']:
            got = run(a, n, axis, op)
            want = oracle.reduce(a, n, axis, op)
            np.testing.assert_array_equal(got, want, err_msg=str((shape, axis, n, op)))


@pytest.mark.parametrize("dtype", ['cf32', 'ci8', 'ci16'])
def test_complex(dtype):
    rng = np.random.default_rng(1234)
    for shape in [(20, 20, 40), (16, 32, 64)]:
        re = ((rng.random(size=shape) * 2 - 1) * 127).astype(np.int8)
        im = ((rng.random(size=shape) * 2 - 1) * 127).astype(np.int8)
        if dtype == 'cf32':
            a = (re + 1j * im).astype(np.complex64)
        else:
            a = np.empty(shape, dtype=bf.DataType(dtype).as_numpy_dtype())
            a['re'], a['im'] = re, im
        for axis in range(3):
            for n in [2, 4, 5, 8, None]:
                if n is not None and shape[axis] % n:
                    continue
                for op in ['sum', 'mean', 'stderr', 'pwrsum', 'pwrmean', 'pwrmin', 'pwrmax']:
                    want = oracle.reduce(a, n, axis, op)
                    got = run(a, n, axis, op, 'f32' if op.startswith('pwr') else 'cf32')
                    np.testing.assert_allclose(got, want, rtol=1e-6, err_msg=str((shape, axis, n, op)))


def test_baseline_config1_and_chain_shapes():
    """BASELINE config 1 (f32 [4096 frames, 256 chan]) and the GUPPI chain's
    reduce (f32 [4, N] -> [4, N/4], vec4 path)."""
    rng = np.random.default_rng(1)
    a = rng.normal(size=(4096, 256)).astype(np.float32)
    np.testing.assert_array_equal(run(a, 4, 1, 'sum'), oracle.reduce(a, 4, 1, 'sum'))
    np.testing.assert_array_equal(run(a, 8, 0, 'sum'), oracle.reduce(a, 8, 0, 'sum'))
    b = rng.normal(size=(4, 1 << 20)).astype(np.float32)
    np.testing.assert_array_equal(run(b, 4, 1, 'sum'), oracle.reduce(b, 4, 1, 'sum'))


def test_errors():
    from bifrost_b200.libbifrost import _bf
    a = bf.empty((8, 8), dtype='f32', space='cuda')
    b = bf.empty((4, 4), dtype='f32', space='cuda')       # two reduced axes
    assert _bf.bfReduce(a.as_BFarray(), b.as_BFarray(), 0) == _bf.BF_STATUS_UNSUPPORTED_SHAPE
    c = bf.empty((8, 3), dtype='f32', space='cuda')       # non-integer factor
    assert _bf.bfReduce(a.as_BFarray(), c.as_BFarray(), 0) == _bf.BF_STATUS_INVALID_SHAPE
    d = bf.empty((8, 8), dtype='f32', space='cuda')       # nothing reduced
    assert _bf.bfReduce(a.as_BFarray(), d.as_BFarray(), 0) == _bf.BF_STATUS_INVALID_SHAPE
    h = bf.empty((8, 4), dtype='f32', space='system')
    assert _bf.bfReduce(a.as_BFarray(), h.as_BFarray(), 0) == _bf.BF_STATUS_UNSUPPORTED_SPACE


def test_reduce_matches_the_reference_library():
    """What the reference's own bfReduce (src/reduce.cu:881-920) computed for the
    same inputs (tests/golden/ref_golden.npz, tests/golden/make_ref_golden.py):
    bit-identical for sum / min / max on float data (same left-to-right order),
    1 ulp for mean."""
    import os
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from golden import digest
    from golden import make_ref_golden as refgold
    g = np.load(refgold.GOLDEN)
    for shape, axis, n, a in refgold.reduce_inputs():
        oshape = list(shape)
        oshape[axis] //= n
        d_a = bf.asarray(a, space='cuda')
        for name in refgold.REDUCE_OPS:
            d_o = bf.empty(oshape, 'f32', 'cuda')
            bf.reduce(d_a, d_o, name)
            ours = np.asarray(d_o.copy('system'))
            key = refgold.reduce_key(shape, axis, n, name)
            if name in refgold.REDUCE_EXACT:
                digest.check(g, key, ours, lambda o, t: np.testing.assert_array_equal(o, t, err_msg=key))
            else:
                digest.check_close(g, key, ours, rtol=2e-7)
