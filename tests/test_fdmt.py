"""FDMT parity.  CPU: the oracle against the golden outputs of the reference's
own CUDA code.  GPU: libbifrost_b200 against the oracle (bit-exact -- the FDMT
is a fixed tree of fp32 operations), against the reference library when it
travelled, plus the reference's own smoke checks (test/test_fdmt.py:38-65) and
size-independent properties at large sizes."""
import ctypes
import os
import sys

import numpy as np
import pytest

import bifrost_b200 as bf
from bifrost_b200.fdmt import Fdmt
from oracle import fdmt as ofdmt

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from golden import digest  # noqa: E402
from golden import make_ref_golden as refgold  # noqa: E402
from golden.make_fdmt_golden import CASES as GOLDEN_CASES, SENTINEL, make_input  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'fdmt_ref_golden.npz')


def assert_same_bits(a, b):
    a = np.ascontiguousarray(a, dtype=np.float32)
    b = np.ascontiguousarray(b, dtype=np.float32)
    assert a.shape == b.shape
    mism = a.view(np.uint32) != b.view(np.uint32)
    both_nan = np.isnan(a) & np.isnan(b)
    mism &= ~both_nan
    assert not mism.any(), f"{mism.sum()} of {mism.size} values differ; first at {np.argwhere(mism)[0]}"


# ------------------------------------------------------------------ CPU ----
@pytest.mark.skipif(not os.path.exists(GOLDEN), reason="golden file not generated yet")
@pytest.mark.parametrize("case", GOLDEN_CASES, ids=[c[0] for c in GOLDEN_CASES])
def test_oracle_matches_reference_golden(case):
    """Pins oracle/fdmt.py against outputs of the reference CUDA library."""
    name, ntime, nchan, md, f0, df, dtype, batch = case
    i = [c[0] for c in GOLDEN_CASES].index(name)
    x = make_input(name, batch + (nchan, ntime), dtype, 1234 + i)
    x = x.astype(np.float32) if dtype == 'f32' else x
    out = np.full(batch + (md, ntime), SENTINEL, np.float32)
    ofdmt.fdmt(x, md, f0, df, out=out)
    digest.check(np.load(GOLDEN), name + '/out', out, assert_same_bits)


def test_oracle_dispersed_pulse_peaks_at_its_dm():
    """A pulse following the nu^-2 law sums to (about) nchan in row d."""
    nchan, ntime, md = 64, 512, 60
    f0, df = 1000., 400. / nchan
    plan = ofdmt.FdmtPlan(nchan, md, f0, df)
    x = np.zeros((nchan, ntime), np.float32)
    d_true, t0 = 41, 100
    fmin, fmax = f0, f0 + (nchan - 1) * df
    for c in range(nchan):
        rel = ((f0 + c * df) ** -2 - fmax ** -2) / (fmin ** -2 - fmax ** -2)
        x[c, t0 + int(round(rel * d_true))] = 1.0
    out = ofdmt.fdmt(x, md, f0, df, plan=plan)
    r, t = np.unravel_index(np.nanargmax(out), out.shape)
    assert abs(r - d_true) <= 1 and abs(t - t0) <= 1
    assert out[r, t] > 0.6 * nchan


# ------------------------------------------------------------------ GPU ----
def run_gpu(x, md, f0, df, batch=(), negative_delays=False, sentinel=SENTINEL, workspace=False):
    nchan, ntime = x.shape[-2:]
    plan = Fdmt()
    plan.init(nchan, md, f0, df, -2.0, 'cuda')
    d_in = bf.asarray(x, space='cuda')
    d_out = bf.asarray(np.full(x.shape[:-2] + (md, ntime), sentinel, np.float32), space='cuda')
    if workspace:
        size = plan.get_workspace_size(d_in, d_out)
        ws = bf.empty((size,), dtype='u8', space='cuda')
        plan.execute_workspace(d_in, d_out, ws.ctypes.data, size, negative_delays)
    else:
        plan.execute(d_in, d_out, negative_delays)
    bf.device.stream_synchronize()
    return np.asarray(d_out.copy('system'))


@pytest.mark.gpu
@pytest.mark.parametrize("case", GOLDEN_CASES, ids=[c[0] for c in GOLDEN_CASES])
def test_gpu_matches_oracle_bit_exact(case):
    name, ntime, nchan, md, f0, df, dtype, batch = case
    i = [c[0] for c in GOLDEN_CASES].index(name)
    x = make_input(name, batch + (nchan, ntime), dtype, 1234 + i)
    x = x.astype(np.float32) if dtype == 'f32' else x
    got = run_gpu(x, md, f0, df)
    want = np.full(batch + (md, ntime), SENTINEL, np.float32)
    ofdmt.fdmt(x, md, f0, df, out=want)
    assert_same_bits(got, want)
    if os.path.exists(GOLDEN):
        digest.check(np.load(GOLDEN), name + '/out', got, assert_same_bits)


@pytest.mark.gpu
@pytest.mark.parametrize("ntime,nchan,md,batch", [
    (1024, 128, 200, ()), (1024, 2, 20, ()), (1024, 32, 2, ()), (1024, 32, 1, ()),
    (1024, 33, 65, ()), (17, 33, 65, ()),
    (1024, 128, 200, (7,)), (1024, 2, 20, (7,)), (1024, 33, 65, (7,)), (17, 33, 65, (7,)),
    (256, 32, 20, (3, 2, 5)), (17, 33, 65, (3, 2, 5)),
])
def test_reference_smoke_semantics(ntime, nchan, md, batch):
    """test/test_fdmt.py:38-65: untouched cells keep the sentinel, values stay
    bounded, execute == execute_workspace bit for bit."""
    rng = np.random.default_rng(1234)
    x = rng.normal(size=batch + (nchan, ntime)).astype(np.float32)
    f0, df = 1000., 400. / nchan
    o1 = run_gpu(x, md, f0, df)
    if md > 1:
        assert o1.min() == SENTINEL
    assert o1.max() < 100.
    o2 = run_gpu(x, md, f0, df, workspace=True)
    np.testing.assert_equal(o1, o2)
    want = np.full(batch + (md, ntime), SENTINEL, np.float32)
    ofdmt.fdmt(x, md, f0, df, out=want)
    assert_same_bits(o1, want)


_OLD = dict(BFB_FDMT_PACKED='0')     # the float schedules: switch the packed-integer schedule off


@pytest.mark.gpu
@pytest.mark.parametrize("knob", [dict(BFB_FDMT_V1='1'), dict(_OLD), dict(_OLD, BFB_FDMT_K='2'),
                                  dict(_OLD, BFB_FDMT_K='4', BFB_FDMT_SMEM_KB='48'),
                                  dict(_OLD, BFB_FDMT_K='8'), dict(_OLD, BFB_FDMT_TAIL_TILE='1024', BFB_FDMT_TAIL_ROWS='3'),
                                  dict(_OLD, BFB_FDMT_THREADS='128'),
                                  dict(_OLD, BFB_FDMT_TILES='0'), dict(_OLD, BFB_FDMT_RAWTILES='0'),
                                  dict(_OLD, BFB_FDMT_TILE_D='8', BFB_FDMT_SPLIT='7,9'),
                                  dict(_OLD, BFB_FDMT_TILE_D='64', BFB_FDMT_TILES_PER_CTA='3'),
                                  dict(_OLD, BFB_FDMT_K='3', BFB_FDMT_TILE_THREADS='128'),
                                  dict(_OLD, BFB_FDMT_K='1', BFB_FDMT_SPLIT='2,3,5,8'),
                                  # packed-integer schedule (fdmt_packed.cuh): default and reshaped,
                                  # pass per launch and as the one persistent kernel
                                  dict(), dict(BFB_FDMT_PACKED_SPLIT='3,6'), dict(BFB_FDMT_PACKED_SPLIT='2,4,6,8'),
                                  dict(BFB_FDMT_PACKED_D='8,8,8', BFB_FDMT_PACKED_SMEM_KB='100,50,40'),
                                  dict(BFB_FDMT_PACKED_WARPS='4,2,1'),
                                  dict(BFB_FDMT_PACKED_TCAP='128,200,64', BFB_FDMT_PACKED_D='5,100,7'),
                                  dict(BFB_FDMT_PACKED_MEGA='1'),
                                  dict(BFB_FDMT_PACKED_MEGA='1', BFB_FDMT_PACKED_CHUNK='300', BFB_FDMT_PACKED_TCAP='128,96,64'),
                                  dict(BFB_FDMT_PACKED_MEGA='1', BFB_FDMT_PACKED_SPLIT='2,4,6,8', BFB_FDMT_PACKED_CHUNK='1000')])
def test_every_schedule_gives_the_same_bits(knob):
    """The step-by-step schedule (v1), the fused head + row-blocked tail (v2),
    the shared-memory tile passes (fdmt_tiles.cuh) and the packed-integer
    schedule (default for 1-byte inputs; fdmt_packed.cuh) at several split
    levels / block sizes must agree bit for bit with the oracle."""
    rng = np.random.default_rng(21)
    old = {k: os.environ.get(k) for k in knob}
    os.environ.update(knob)
    try:
        for (ntime, nchan, md, dtype, f0, bw) in [
                (3000, 300, 150, np.int8, 1100., 300.), (5000, 64, 40, np.float32, 1100., 300.),
                (700, 1024, 90, np.uint8, 1100., 300.), (2500, 37, 33, np.int16, 1100., 300.),
                # wide fractional band: step-0 rows with more than 4 delays (exact path of the raw pass)
                (2000, 48, 400, np.int8, 60., 30.), (1500, 21, 300, np.uint8, 40., 25.)]:
            if dtype == np.float32:
                x = rng.normal(size=(nchan, ntime)).astype(np.float32)
            elif dtype == np.int8:
                x = rng.integers(-128, 128, size=(nchan, ntime)).astype(dtype)
            else:
                x = rng.integers(0, 256 if dtype == np.uint8 else 100, size=(nchan, ntime)).astype(dtype)
            df = bw / nchan
            got = run_gpu(x, md, f0, df)
            want = np.full((md, ntime), SENTINEL, np.float32)
            ofdmt.fdmt(x, md, f0, df, out=want)
            assert_same_bits(got, want)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


@pytest.mark.gpu
def test_negative_delays_match_oracle():
    """negative_delays mirrors time as the reference does (src/fdmt.cu:80-81,
    150-151, 702-708); cells whose reference value depends on an out-of-bounds
    read are excluded (documented divergence: we contribute 0 there)."""
    rng = np.random.default_rng(22)
    for (ntime, nchan, md) in [(600, 64, 40), (1000, 48, 30)]:
        x = rng.integers(-50, 50, size=(nchan, ntime)).astype(np.int8)
        f0, df = 1000., 400. / nchan
        got = run_gpu(x, md, f0, df, negative_delays=True)
        want = np.full((md, ntime), SENTINEL, np.float32)
        ofdmt.fdmt(x, md, f0, df, negative_delays=True, out=want)
        assert_same_bits(got, want)


@pytest.mark.gpu
def test_gpu_matches_reference_library():
    """Bit for bit what the reference's own bfFdmtExecute computed for the same
    inputs (tests/golden/ref_golden.npz, tests/golden/make_ref_golden.py)."""
    g = np.load(refgold.GOLDEN)
    for ntime, nchan, md, x in refgold.fdmt_inputs():
        got = run_gpu(x, md, 1000., 400. / nchan)
        digest.check(g, refgold.fdmt_key(ntime, nchan, md, x), got, assert_same_bits)


@pytest.mark.gpu
def test_ring_style_padded_strides():
    """Input rows with a pitch >> ntime and a batch (pol) axis, as handed over
    by a ring span (SURVEY 8b layout fact 1)."""
    rng = np.random.default_rng(3)
    npol, nchan, ntime, pitch, md = 2, 48, 500, 1024, 30
    base = rng.integers(-100, 100, size=(npol, nchan, pitch)).astype(np.int8)
    d_base = bf.asarray(base, space='cuda')
    d_in = d_base[:, :, 7:7 + ntime]
    obase = bf.asarray(np.full((npol, md, pitch), SENTINEL, np.float32), space='cuda')
    d_out = obase[:, :, :ntime]
    f0, df = 1200., 2.0
    plan = Fdmt()
    plan.init(nchan, md, f0, df)
    plan.execute(d_in, d_out)
    bf.device.stream_synchronize()
    got = np.asarray(obase.copy('system'))
    want = np.full((npol, md, ntime), SENTINEL, np.float32)
    ofdmt.fdmt(base[:, :, 7:7 + ntime], md, f0, df, out=want)
    assert_same_bits(got[:, :, :ntime], want)
    assert (got[:, :, ntime:] == SENTINEL).all()


@pytest.mark.gpu
def test_large_gulp_properties():
    """Size-independent checks at a BASELINE-like size (oracle too slow here):
    (1) a dispersed pulse lands in its DM row with ~nchan amplitude,
    (2) linearity: fdmt(a + b) == fdmt(a) + fdmt(b) for integer-valued data
        small enough that every partial sum is exact in fp32 before scaling,
    (3) time-shift covariance away from the edges."""
    nchan, ntime, md = 1024, 32768, 400
    f0, df = 1000., 400. / nchan
    fmax = f0 + (nchan - 1) * df
    x = np.zeros((nchan, ntime), np.int8)
    d_true, t0 = 333, 5000
    for c in range(nchan):
        rel = ((f0 + c * df) ** -2 - fmax ** -2) / (f0 ** -2 - fmax ** -2)
        x[c, t0 + int(round(rel * d_true))] = 1
    out = run_gpu(x, md, f0, df, sentinel=0.0)
    r, t = np.unravel_index(np.argmax(out), out.shape)
    assert abs(r - d_true) <= 1 and abs(t - t0) <= 1
    assert out[r, t] > 0.5 * nchan
    x2 = np.roll(x, 1000, axis=1)
    out2 = run_gpu(x2, md, f0, df, sentinel=0.0)
    np.testing.assert_array_equal(out2[:, 2000:ntime - md], out[:, 1000:ntime - md - 1000])


@pytest.mark.gpu
@pytest.mark.parametrize("md,f0,bw", [(204, 1000., 400.), (794, 1000., 400.), (1621, 1200., 300.)])
def test_schedules_agree_bit_for_bit_at_baseline_sizes(md, f0, bw):
    """BASELINE config 2 geometry (4096 channels; max_delay 204 / 794 / 1621 as in
    SURVEY 8d) on a shortened gulp: the default tile-pass schedule must give the
    same bits as the step-by-step schedule, which the small cases pin against the
    oracle and the reference's own kernels."""
    nchan, ntime = 4096, 6000 + md
    rng = np.random.default_rng(md)
    x = np.clip(np.rint(rng.normal(0, 20, size=(nchan, ntime))), -127, 127).astype(np.int8)
    got = run_gpu(x, md, f0, bw / nchan)
    os.environ['BFB_FDMT_V1'] = '1'
    try:
        want = run_gpu(x, md, f0, bw / nchan)
    finally:
        os.environ.pop('BFB_FDMT_V1', None)
    assert_same_bits(got, want)


def _oracle_windows(x, md, f0, df, got, windows):
    """Compares output columns [a, a+w) of a long gulp with the C oracle run on
    the input slice those columns depend on (columns a .. a+w+md: row r at
    column c sums input times c .. c+r).  The slice's own t < 0 edge never
    reaches the compared columns except for a == 0, where it is the gulp's."""
    from oracle import fdmt_c
    assert fdmt_c.available()
    nchan, ntime = x.shape
    plan = fdmt_c.Plan(nchan, md, f0, df)
    for a, w in windows:
        b = min(ntime, a + w + md)
        xs = np.ascontiguousarray(x[:, a:b])
        want = np.full((md, b - a), SENTINEL, np.float32)
        plan.execute(xs, want)
        n = min(w, b - a)
        # cells the reference leaves unwritten (column >= ntime - r) exist only in
        # the window that touches the end of the gulp; there both hold the sentinel
        assert_same_bits(got[:, a:a + n], want[:, :n])


@pytest.mark.gpu
@pytest.mark.parametrize("md,f0,bw", [(794, 1000., 400.), (204, 1000., 400.), (1621, 1200., 300.)])
def test_baseline_gulp_matches_the_oracle_at_full_size(md, f0, bw):
    """VALUE check of the exact gulp bench.py times (BASELINE config 2: 4096 chan x
    131072+max_delay int8 with the three injected pulses; plus SURVEY 8d's
    max_delay 204 / 1621 variants): five disjoint 8192-column windows, both
    edges included, bit for bit against oracle/fdmt_c.c."""
    import bench
    nchan = 4096
    w = dict(nchan=nchan, ntime=131072 + md, max_delay=md, f0=f0, df=bw / nchan)
    x = bench.make_input(w, 1234)
    got = run_gpu(x, md, f0, bw / nchan)
    ntime = w['ntime']
    wins = [(0, 8192), (40000, 8192), (65536 + 3, 8192), (100001, 8192), (ntime - 8192 - md, 8192 + md)]
    _oracle_windows(x, md, f0, bw / nchan, got, wins)
    if md == 794:
        # the injected pulses come out in their DM rows
        for frac, t0 in ((0.2, ntime // 5), (0.5, ntime // 2), (0.9, (3 * ntime) // 4)):
            d = int(round(frac * (md - 1)))
            blk = got[max(0, d - 2):d + 3, t0 - 3:t0 + 4]
            assert blk.max() > 0.5 * 100 * nchan


def test_plan_that_leaves_its_parent_band_is_rejected():
    """nchan=256, max_delay=300 at 1000-1400 MHz makes a source row index fall
    outside its parent band (step 7); the reference hits assert() and aborts
    (src/fdmt.cu:513-514).  Here it is a status, not a crash."""
    from bifrost_b200.libbifrost import _bf
    n = ctypes.c_int()
    assert _bf.bfFdmtPlanQuery(256, 300, 1000., 400. / 256, -2.0, -1, ctypes.byref(n), None) == \
        _bf.BF_STATUS_INTERNAL_ERROR


@pytest.mark.gpu
def test_status_codes():
    from bifrost_b200.libbifrost import _bf
    plan = Fdmt()
    plan.init(16, 8, 1000., 10.)
    bad_in = bf.empty((15, 64), dtype='f32', space='cuda')
    out = bf.empty((8, 64), dtype='f32', space='cuda')
    assert _bf.bfFdmtExecute(plan.obj, bad_in.as_BFarray(), out.as_BFarray(), 0, None, None) == \
        _bf.BF_STATUS_INVALID_SHAPE
    good_in = bf.empty((16, 64), dtype='f32', space='cuda')
    small = _bf.BFsize(16)
    ws = bf.empty((16,), dtype='u8', space='cuda')
    assert _bf.bfFdmtExecute(plan.obj, good_in.as_BFarray(), out.as_BFarray(), 0,
                             ws.ctypes.data, ctypes.byref(small)) == \
        _bf.BF_STATUS_INSUFFICIENT_STORAGE
    host_in = bf.empty((16, 64), dtype='f32', space='system')
    assert _bf.bfFdmtExecute(plan.obj, host_in.as_BFarray(), out.as_BFarray(), 0, None, None) == \
        _bf.BF_STATUS_UNSUPPORTED_SPACE
