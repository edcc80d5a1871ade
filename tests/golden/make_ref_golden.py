"""Generates tests/golden/ref_golden.npz: what the REFERENCE's own CUDA library
(oracle/_ref/libbifrost_ref.so, built by oracle/ref_build.sh) computes for the
seeded inputs of the tests that compare with it -- bfReduce
(tests/test_reduce.py), the correlator bfLinAlgMatMul (tests/test_linalg.py),
bfQuantize to packed sub-byte types (tests/test_quantize.py) and bfFdmtExecute
(tests/test_fdmt.py).  Needs a B200 and the reference library:

    python tests/golden/make_ref_golden.py OUT.npz

then copy OUT.npz to tests/golden/ref_golden.npz.  Outputs too large to store
whole keep a digest and a sample (tests/golden/digest.py).
"""
import ctypes
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from golden import digest  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'ref_golden.npz')

# (shape, axis, factor); sum / min / max / pwrsum are bit-identical, mean to 1 ulp
REDUCE_CASES = [((4096, 256), 1, 4), ((4096, 256), 0, 8), ((4, 65536), 1, 4), ((20, 40, 60), 1, 5)]
REDUCE_OPS = ['sum', 'min', 'max', 'mean', 'pwrsum']
REDUCE_EXACT = ('sum', 'min', 'max', 'pwrsum')
# (ntime, nchan, nstand*npol); the reference is exact only for short integrations
LINALG_CASES = [(64, 3, 32), (512, 4, 512), (200, 2, 130)]
LINALG_EXACT_NTIME = 64
# (odtype, nbit) x scale
QUANTIZE_CASES = [(o, b, s) for s in (1.0, 0.37)
                  for (o, b) in [('i4', 4), ('ci4', 4), ('i2', 2), ('ci2', 2), ('i1', 1), ('ci1', 1)]]
# (ntime, nchan, max_delay, dtype); f0 = 1000 MHz, bw = 400 MHz
FDMT_CASES = [(2000, 256, 301, np.float32), (1500, 100, 64, np.int8),
              (4096, 512, 130, np.int8), (333, 17, 40, np.uint16)]
FDMT_SENTINEL = -999.0


def reduce_inputs():
    rng = np.random.default_rng(11)
    for shape, axis, n in REDUCE_CASES:
        yield shape, axis, n, rng.normal(size=shape).astype(np.float32)


def reduce_key(shape, axis, n, op):
    return 'reduce/%s_a%d_n%d/%s' % ('x'.join(map(str, shape)), axis, n, op)


def linalg_inputs():
    from test_linalg import rand_ci8
    rng = np.random.default_rng(77)
    for ntime, nchan, n in LINALG_CASES:
        yield ntime, nchan, n, rand_ci8(rng, (ntime, nchan, n))


def linalg_key(ntime, nchan, n):
    return 'linalg/t%d_c%d_n%d' % (ntime, nchan, n)


def quantize_key(odtype, scale):
    return 'quantize/%s_s%g' % (odtype, scale)


def fdmt_inputs():
    rng = np.random.default_rng(7)
    for ntime, nchan, md, dtype in FDMT_CASES:
        if dtype == np.float32:
            x = rng.normal(size=(nchan, ntime)).astype(np.float32)
        else:
            info = np.iinfo(dtype)
            x = rng.integers(max(info.min, -127), min(info.max, 127) + 1, size=(nchan, ntime)).astype(dtype)
        yield ntime, nchan, md, x


def fdmt_key(ntime, nchan, md, x):
    return 'fdmt/t%d_c%d_d%d_%s' % (ntime, nchan, md, x.dtype.name)


def main(out_path):
    import bifrost_b200 as bf
    from bifrost_b200.libbifrost import _bf, _check
    import reflib
    ref = reflib.load()
    assert ref is not None, 'oracle/_ref/libbifrost_ref.so missing: run oracle/ref_build.sh'
    store = {}

    codes = dict(sum=_bf.BF_REDUCE_SUM, min=_bf.BF_REDUCE_MIN, max=_bf.BF_REDUCE_MAX,
                 mean=_bf.BF_REDUCE_MEAN, pwrsum=_bf.BF_REDUCE_POWER_SUM)
    for shape, axis, n, a in reduce_inputs():
        oshape = list(shape)
        oshape[axis] //= n
        d_a = bf.asarray(a, space='cuda')
        for op in REDUCE_OPS:
            d_r = bf.empty(oshape, 'f32', 'cuda')
            _check(ref.bfReduce(d_a.as_BFarray(), d_r.as_BFarray(), codes[op]))
            _check(ref.bfStreamSynchronize())
            store.update(digest.pack(reduce_key(shape, axis, n, op), np.asarray(d_r.copy('system')),
                                     exact=op in REDUCE_EXACT))

    for ntime, nchan, n, x in linalg_inputs():
        d_x = bf.asarray(x, space='cuda')
        d_c = bf.zeros((nchan, n, n), 'cf32', 'cuda')
        h = ctypes.c_void_p()
        _check(ref.bfLinAlgCreate(ctypes.byref(h)))
        _check(ref.bfLinAlgMatMul(h, 1.0, None, d_x.transpose((1, 0, 2)).as_BFarray(), 0.0, d_c.as_BFarray()))
        _check(ref.bfStreamSynchronize())
        _check(ref.bfLinAlgDestroy(h))
        c = np.asarray(d_c.copy('system'))
        il = np.tril_indices(n)
        store.update(digest.pack(linalg_key(ntime, nchan, n), c[:, il[0], il[1]],
                                 exact=ntime <= LINALG_EXACT_NTIME))

    from test_quantize import _packed_case
    for odtype, nbit, scale in QUANTIZE_CASES:
        cplx = odtype.startswith('c')
        x = _packed_case(nbit, cplx)
        d_in = bf.asarray(x, space='cuda')
        nbyte = x.size * (2 if cplx else 1) * nbit // 8
        d_raw = bf.asarray(np.zeros(nbyte, np.uint8), space='cuda')
        d_out = bf.ndarray(space='cuda', buffer=d_raw.ctypes.data, shape=x.shape, dtype=odtype)
        # (the reference's contiguity test rejects the byte strides of real
        # sub-byte arrays -- BF_STATUS_UNSUPPORTED_STRIDE; the complex ones go through)
        status = ref.bfQuantize(d_in.as_BFarray(), d_out.as_BFarray(), float(scale))
        store[quantize_key(odtype, scale) + '/status'] = np.array(status)
        if status == 0:
            _check(ref.bfStreamSynchronize())
            store[quantize_key(odtype, scale) + '/bytes'] = np.asarray(d_raw.copy('system'))

    for ntime, nchan, md, x in fdmt_inputs():
        f0, df = 1000., 400. / nchan
        d_in = bf.asarray(x, space='cuda')
        d_out = bf.asarray(np.full((md, ntime), FDMT_SENTINEL, np.float32), space='cuda')
        plan = ctypes.c_void_p()
        _check(ref.bfFdmtCreate(ctypes.byref(plan)))
        _check(ref.bfFdmtInit(plan, nchan, md, f0, df, -2.0, 2, None, None))
        _check(ref.bfFdmtExecute(plan, d_in.as_BFarray(), d_out.as_BFarray(), 0, None, None))
        _check(ref.bfStreamSynchronize())
        _check(ref.bfFdmtDestroy(plan))
        store.update(digest.pack(fdmt_key(ntime, nchan, md, x), np.asarray(d_out.copy('system')), exact=True))

    np.savez_compressed(out_path, **store)
    print('wrote', out_path, os.path.getsize(out_path), 'bytes')


if __name__ == '__main__':
    main(sys.argv[1] if len(sys.argv) > 1 else GOLDEN)
