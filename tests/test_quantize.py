"""bfQuantize: the reference's known answers (test/test_quantize.py:33-50) and
random data against the oracle, bit-exact."""
import numpy as np
import pytest

import bifrost_b200 as bf
from oracle import quantize as oquant

KNOWN_IN = np.array([[0.4 + 0.5j, 1.4 + 1.5j], [2.4 + 2.5j, 3.4 + 3.5j], [4.4 + 4.5j, 5.4 + 5.5j]], np.complex64)
KNOWN_OUT = np.array([[(0, 0), (1, 2)], [(2, 2), (3, 4)], [(4, 4), (5, 6)]])


@pytest.mark.parametrize("kind", ['i8', 'i16', 'i32'])
def test_oracle_reproduces_reference_known_answers(kind):
    np.testing.assert_array_equal(oquant.quantize(KNOWN_IN, kind), KNOWN_OUT)


@pytest.mark.gpu
@pytest.mark.parametrize("odtype", ['ci8', 'ci16', 'ci32'])
def test_gpu_known_answers(odtype):
    d_in = bf.asarray(KNOWN_IN, space='cuda')
    d_out = bf.empty((3, 2), dtype=odtype, space='cuda')
    bf.quantize(d_in, d_out)
    out = np.asarray(d_out.copy('system'))
    np.testing.assert_array_equal(np.stack([out['re'], out['im']], -1), KNOWN_OUT)


@pytest.mark.gpu
@pytest.mark.parametrize("odtype", ['i8', 'i16', 'i32', 'u8', 'u16', 'u32', 'ci8', 'ci16'])
@pytest.mark.parametrize("scale", [1.0, 0.37, 1e6])
def test_gpu_matches_oracle(odtype, scale):
    rng = np.random.default_rng(5)
    n = 100003
    cplx = odtype.startswith('c')
    x = (rng.normal(size=n) * 300).astype(np.float32)
    x[:8] = [0.5, 1.5, 2.5, -0.5, -1.5, 1e20, -1e20, 127.5]
    if odtype.endswith('32'):
        x[5:7] = [1e3, -1e3]          # saturation of 32-bit outputs is undefined in the reference
    if cplx:
        x = (x + 1j * (rng.normal(size=n) * 300).astype(np.float32)).astype(np.complex64)
    d_out = bf.empty((n,), dtype=odtype, space='cuda')
    bf.quantize(bf.asarray(x, space='cuda'), d_out, scale)
    out = np.asarray(d_out.copy('system'))
    got = np.stack([out['re'], out['im']], -1) if cplx else out
    np.testing.assert_array_equal(got, oquant.quantize(x, odtype.lstrip('c'), scale))


@pytest.mark.gpu
def test_status_codes():
    from bifrost_b200.libbifrost import _bf
    a = bf.empty((4,), 'f32', 'cuda')
    b = bf.empty((5,), 'i8', 'cuda')
    c = bf.empty((4,), 'ci8', 'cuda')
    assert _bf.bfQuantize(a.as_BFarray(), b.as_BFarray(), 1.0) == _bf.BF_STATUS_INVALID_SHAPE
    assert _bf.bfQuantize(a.as_BFarray(), c.as_BFarray(), 1.0) == _bf.BF_STATUS_INVALID_DTYPE


# ---- sub-byte outputs (src/guantize.cu:146-348) --------------------------------
def test_packed_oracle_layout():
    """First value in the most significant bits; 4-bit clips to +-7, 2-bit to +-1."""
    assert oquant.quantize_packed(np.array([1.2, -2.6], np.float32), 4).tolist() == [0x1D]
    assert oquant.quantize_packed(np.array([9.0, -9.0], np.float32), 4).tolist() == [0x79]
    assert oquant.quantize_packed(np.array([0.4, -0.6, 3.0, 0.5], np.float32), 2).tolist() == [0b00110100]
    assert oquant.quantize_packed(np.array([1, -1, 0, -0.0, 5, -5, -2, 3], np.float32), 1).tolist() == [0b10111001]


def _packed_case(nbit, cplx, n=4096 * 8 + 24):
    rng = np.random.default_rng(nbit * 2 + cplx)
    x = (rng.normal(size=n) * (4.0 if nbit == 4 else 1.0)).astype(np.float32)
    x[:8] = [0.5, 1.5, 2.5, -0.5, -1.5, 1e20, -1e20, 6.5]
    if cplx:
        x = (x[0::2] + 1j * x[1::2]).astype(np.complex64)
    return x


@pytest.mark.gpu
@pytest.mark.parametrize("odtype,nbit", [('i4', 4), ('ci4', 4), ('i2', 2), ('ci2', 2), ('i1', 1), ('ci1', 1)])
@pytest.mark.parametrize("scale", [1.0, 0.37])
def test_gpu_packed_outputs_match_oracle_and_reference(odtype, nbit, scale):
    import sys, os
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from golden import make_ref_golden as refgold
    cplx = odtype.startswith('c')
    x = _packed_case(nbit, cplx)
    d_in = bf.asarray(x, space='cuda')
    nbyte = x.size * (2 if cplx else 1) * nbit // 8
    d_raw = bf.asarray(np.zeros(nbyte, np.uint8), space='cuda')
    d_out = bf.ndarray(space='cuda', buffer=d_raw.ctypes.data, shape=x.shape, dtype=odtype)
    bf.quantize(d_in, d_out, scale)
    got = np.asarray(d_raw.copy('system'))
    want = oquant.quantize_packed(x, nbit, scale)
    np.testing.assert_array_equal(got, want)
    # what the reference's own GPU kernels wrote for the same input
    # (tests/golden/make_ref_golden.py; 1-bit: on the bits its masks keep -- see
    # oracle/quantize.py).  The reference's contiguity test rejects the byte
    # strides of every packed type here but ci4 (BF_STATUS_UNSUPPORTED_STRIDE,
    # stored as the status): for those there is nothing to compare.
    g = np.load(refgold.GOLDEN)
    key = refgold.quantize_key(odtype, scale)
    if int(g[key + '/status']) == 0:
        theirs = g[key + '/bytes']
        mask = oquant.reference_1bit_mask if nbit == 1 else 0xFF
        np.testing.assert_array_equal(got & mask, theirs & mask)


@pytest.mark.gpu
@pytest.mark.parametrize("odtype,nbit", [('ci4', 4), ('i2', 2), ('i4', 4)])
def test_gpu_quantize_then_unpack_round_trip(odtype, nbit):
    """unpack(quantize(x)) == clip(rint(x)): the packed layout is the one bfUnpack
    reads as big-endian sub-words (first value in the high bits)."""
    cplx = odtype.startswith('c')
    x = _packed_case(nbit, cplx, 4096)
    d_in = bf.asarray(x, space='cuda')
    nval = x.size * (2 if cplx else 1)
    d_raw = bf.asarray(np.zeros(nval * nbit // 8, np.uint8), space='cuda')
    d_q = bf.ndarray(space='cuda', buffer=d_raw.ctypes.data, shape=x.shape, dtype=odtype, native=False)
    bf.quantize(d_in, d_q)
    d_u = bf.empty(x.shape, dtype='ci8' if cplx else 'i8', space='cuda')
    bf.unpack(d_q, d_u)
    out = np.asarray(d_u.copy('system'))
    got = np.stack([out['re'], out['im']], -1).reshape(-1) if cplx else out
    lim = 7 if nbit == 4 else 1
    v = np.stack([x.real, x.imag], -1).reshape(-1) if cplx else x
    np.testing.assert_array_equal(got, np.rint(np.clip(v, -lim, lim)).astype(np.int8))
