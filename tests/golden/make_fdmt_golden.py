"""Generates tests/golden/fdmt_ref_golden.npz by running the REFERENCE's own
CUDA FDMT (oracle/_ref/libbifrost_ref.so, built by oracle/ref_build.sh) on
seeded inputs.  Needs a GPU:

    python tests/golden/make_fdmt_golden.py OUT.npz

then copy OUT.npz to tests/golden/fdmt_ref_golden.npz.  The reference's tests
hold no FDMT known-answer vector (test/test_fdmt.py:49-65 is a smoke test), so
these outputs are what pins the oracle (oracle/fdmt.py) for this op.  Each
output is stored as its digest and a sample (tests/golden/digest.py); the
inputs are regenerated from their seeds by make_input().
"""
import ctypes
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

# (name, ntime, nchan, max_delay, f0, df, dtype, batch)  -- test/test_fdmt.py:66-103 shapes
CASES = [
    ('t1024_c128_d200', 1024, 128, 200, 1000., 400. / 128, 'f32', ()),
    ('t1024_c2_d20', 1024, 2, 20, 1000., 400. / 2, 'f32', ()),
    ('t1024_c32_d2', 1024, 32, 2, 1000., 400. / 32, 'f32', ()),
    ('t1024_c32_d1', 1024, 32, 1, 1000., 400. / 32, 'f32', ()),
    ('t1024_c33_d65', 1024, 33, 65, 1000., 400. / 33, 'f32', ()),
    ('t17_c33_d65', 17, 33, 65, 1000., 400. / 33, 'f32', ()),
    ('t300_c33_d65_b3', 300, 33, 65, 1000., 400. / 33, 'f32', (3,)),
    ('t777_c64_d90_i8', 777, 64, 90, 1000., 400. / 64, 'i8', ()),
    ('t512_c50_d40_u8_revband', 512, 50, 40, 1400., -4.0, 'u8', ()),
    ('t640_c256_d100_i16', 640, 256, 100, 1200., 300. / 256, 'i16', ()),
]
SENTINEL = -999.0


def make_input(name, shape, dtype, seed):
    rng = np.random.default_rng(seed)
    if dtype == 'f32':
        return rng.normal(size=shape).astype(np.float16)      # stored as f16, used as f32
    if dtype == 'i8':
        return np.clip(np.rint(rng.normal(0, 20, size=shape)), -127, 127).astype(np.int8)
    if dtype == 'u8':
        return rng.integers(0, 256, size=shape).astype(np.uint8)
    if dtype == 'i16':
        return np.rint(rng.normal(0, 3000, size=shape)).astype(np.int16)
    raise ValueError(dtype)


def main(out_path):
    import bifrost_b200 as bf
    from bifrost_b200.libbifrost import _check
    from golden import digest
    import reflib
    ref = reflib.load()
    assert ref is not None, "oracle/_ref/libbifrost_ref.so missing: run oracle/ref_build.sh"
    store = {}
    for i, (name, ntime, nchan, md, f0, df, dtype, batch) in enumerate(CASES):
        x = make_input(name, batch + (nchan, ntime), dtype, 1234 + i)
        xin = x.astype(np.float32) if dtype == 'f32' else x
        d_in = bf.asarray(xin, space='cuda')
        d_out = bf.asarray(np.full(batch + (md, ntime), SENTINEL, np.float32), space='cuda')
        plan = ctypes.c_void_p()
        _check(ref.bfFdmtCreate(ctypes.byref(plan)))
        _check(ref.bfFdmtInit(plan, nchan, md, f0, df, -2.0, 2, None, None))
        _check(ref.bfFdmtExecute(plan, d_in.as_BFarray(), d_out.as_BFarray(), 0, None, None))
        _check(ref.bfStreamSynchronize())
        bf.device.stream_synchronize()
        out = d_out.copy('system')
        _check(ref.bfFdmtDestroy(plan))
        store.update(digest.pack(name + '/out', np.asarray(out), exact=True))
        print(name, 'ok', np.asarray(out).shape)
    np.savez_compressed(out_path, **store)
    print('wrote', out_path)


if __name__ == '__main__':
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(os.path.abspath(__file__)),
                                                            'fdmt_ref_golden.npz'))
