"""bfRing* / bfProcLog* / bfAffinity* of libbifrost_b200.so (csrc/ring.cpp)
against the reference's own ring.

Parity is pinned by tests/golden/ring_traces.json.gz: random scripts of calls
with the answers the reference's unmodified src/ring_impl.cpp gave
(tests/golden/make_ring_golden.py), replayed here call by call, no reference
needed.  When oracle/_ref/libbifrost_ref_ring.so is present (built by
oracle/ref_ring_build.sh), the stored answers and the threaded expectations
below are also checked against the reference's ring itself.
The remaining tests exercise what a single-threaded script cannot: blocking
calls between threads, and rings in device memory (-m gpu).
"""
import ctypes
import gzip
import json
import os
import threading

import numpy as np
import pytest

import ringtrace as rt
from bifrost_b200.libbifrost import _bf, _check, _get, BFspan_info, BFsequence_info, EndOfDataStop

HERE = os.path.dirname(os.path.abspath(__file__))
OURS = rt.load_ours()
REF = rt.load_reference()
needs_ref = pytest.mark.skipif(REF is None, reason='oracle/_ref/libbifrost_ref_ring.so not built')


def golden_cases(key='cases'):
    with gzip.open(os.path.join(HERE, 'golden', 'ring_traces.json.gz')) as f:
        return json.loads(f.read().decode())[key]


def assert_same_trace(script, want, got):
    for i, (op, a, b) in enumerate(zip(script, want, got)):
        assert a == b, f'call {i} {op}: reference {a}, ours {b}; previous calls: {script[max(0, i - 5):i]}'
    assert len(want) == len(got)


@pytest.mark.timeout(120)
@pytest.mark.parametrize('case', golden_cases(), ids=lambda c: 'seed%d' % c['seed'])
def test_replays_the_reference_traces(case):
    got = rt.replay(OURS, case['script'])
    assert_same_trace(case['script'], case['trace'], got)


@needs_ref
@pytest.mark.timeout(120)
def test_golden_traces_are_what_the_reference_does():
    case = golden_cases()[0]
    assert rt.replay(REF, case['script']) == case['trace']


@pytest.mark.timeout(300)
@pytest.mark.parametrize('seed', range(100, 112))
def test_live_differential_against_the_reference_ring(seed):
    """Longer random scripts, built adaptively against the reference's ring
    (ringtrace.generate) and stored with its answers."""
    case, = [c for c in golden_cases('differential') if c['seed'] == seed]
    script, want = case['script'], case['trace']
    assert len(script) > 100
    assert_same_trace(script, want, rt.replay(OURS, script))


# --------------------------------------------------------------------------
# small binding for the threaded tests; `L` is the library under test -- ours,
# or (fixture `lib`) the reference's own ring, so that what these tests expect
# is checked to be the reference's behaviour too
# --------------------------------------------------------------------------
class _Lib(object):
    target = OURS

    def __getattr__(self, name):
        return getattr(_Lib.target, name)


L = _Lib()


@pytest.fixture(params=['ours', 'reference'])
def lib(request):
    if request.param == 'reference':
        if REF is None:
            pytest.skip('oracle/_ref/libbifrost_ref_ring.so not built')
        _Lib.target = REF
    yield request.param
    _Lib.target = OURS


class Ring(object):
    def __init__(self, name, space='system'):
        self.obj = ctypes.c_void_p()
        self.space = _bf.BF_SPACE_CUDA if space == 'cuda' else _bf.BF_SPACE_SYSTEM
        _check(L.bfRingCreate(ctypes.byref(self.obj), name.encode(), self.space))

    def destroy(self):
        _check(L.bfRingDestroy(self.obj))

    def reserve(self, nbyte, nonblocking=False):
        h = ctypes.c_void_p()
        _check(L.bfRingSpanReserve(ctypes.byref(h), self.obj, nbyte, nonblocking))
        return h

    @staticmethod
    def info(span):
        inf = BFspan_info()
        _check(L.bfRingSpanGetInfo(span, ctypes.byref(inf)))
        return inf

    def begin_sequence(self, name, time_tag, header=b'', nringlet=1):
        h = ctypes.c_void_p()
        buf = ctypes.create_string_buffer(header, len(header))
        _check(L.bfRingSequenceBegin(ctypes.byref(h), self.obj, name.encode(), time_tag, len(header),
                                       ctypes.cast(buf, ctypes.c_void_p), nringlet, 0))
        return h

    def open_earliest(self, guarantee=True):
        h = ctypes.c_void_p()
        _check(L.bfRingSequenceOpenEarliest(ctypes.byref(h), self.obj, guarantee))
        return h


def payload(i, r, nbyte):
    return ((np.arange(nbyte, dtype=np.uint32) * 7 + i * 13 + r * 101) & 0xFF).astype(np.uint8)


def span_view(inf, r):
    """numpy view of ringlet r of a system-space span."""
    buf = (ctypes.c_uint8 * inf.size).from_address(inf.data + r * inf.stride)
    return np.frombuffer(buf, dtype=np.uint8)


@pytest.mark.timeout(120)
def test_writer_and_guaranteed_readers_stream_through_a_small_ring(lib):
    """200 gulps through a ring that holds 4: the writer blocks on the slowest
    guaranteed reader, readers block on the writer, spans wrap through the ghost
    region, two sequences, every byte of both ringlets arrives in order."""
    gulp, ngulp, nringlet = 1000, 200, 2
    ring = Ring('threaded')
    _check(L.bfRingResize(ring.obj, gulp, 4 * gulp, nringlet))
    errors = []
    opened = threading.Semaphore(0)

    def writer():
        try:
            _check(L.bfRingBeginWriting(ring.obj))
            i = 0
            for s in range(2):
                seq = ring.begin_sequence('obs%d' % s, 100 + s, b'hdr%d' % s, nringlet)
                if s == 0:
                    for _ in range(2):              # both readers hold their guarantee before data flows
                        assert opened.acquire(timeout=60)
                for _ in range(ngulp // 2):
                    span = ring.reserve(gulp)
                    inf = ring.info(span)
                    assert inf.size == gulp and inf.nringlet == nringlet
                    for r in range(nringlet):
                        span_view(inf, r)[:] = payload(i, r, gulp)
                    _check(L.bfRingSpanCommit(span, gulp))
                    i += 1
                _check(L.bfRingSequenceEnd(seq, 0))
            _check(L.bfRingEndWriting(ring.obj))
        except Exception as e:      # pragma: no cover
            errors.append(e)

    def reader(read_size):
        try:
            seq = ring.open_earliest(guarantee=True)
            opened.release()
            i = 0
            for s in range(2):
                assert _get(L.bfRingSequenceGetName, seq) == b'obs%d' % s
                if hasattr(_Lib.target, 'bfRingSequenceGetInfo'):      # (declared but not defined by the reference)
                    sinf = BFsequence_info()
                    _check(L.bfRingSequenceGetInfo(seq, ctypes.byref(sinf)))
                    assert ctypes.string_at(sinf.header, sinf.header_size) == b'hdr%d' % s and sinf.time_tag == 100 + s
                assert _get(L.bfRingSequenceGetTimeTag, seq) == 100 + s
                offset = 0
                while True:
                    span = ctypes.c_void_p()
                    try:
                        _check(L.bfRingSpanAcquire(ctypes.byref(span), seq, offset, read_size))
                    except EndOfDataStop:
                        break
                    inf = ring.info(span)
                    assert inf.offset == offset and 0 < inf.size <= read_size
                    assert _get(L.bfRingSpanGetSizeOverwritten, span) == 0
                    for r in range(nringlet):
                        got = span_view(inf, r)
                        for j in range(0, inf.size, gulp):
                            np.testing.assert_array_equal(got[j:j + gulp], payload(i + j // gulp, r, gulp)[:inf.size - j])
                    _check(L.bfRingSpanRelease(span))
                    offset += inf.size
                    i += inf.size // gulp
                assert offset == (ngulp // 2) * gulp
                if s == 0:
                    _check(L.bfRingSequenceNext(seq))
            with pytest.raises(EndOfDataStop):
                _check(L.bfRingSequenceNext(seq))
            _check(L.bfRingSequenceClose(seq))
        except Exception as e:      # pragma: no cover
            errors.append(e)

    threads = [threading.Thread(target=reader, args=(gulp,)), threading.Thread(target=reader, args=(gulp,)),
               threading.Thread(target=writer)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(100)
    assert not any(t.is_alive() for t in threads), 'deadlock'
    assert not errors, errors
    ring.destroy()


@pytest.mark.timeout(60)
def test_blocking_reserve_waits_for_the_guaranteed_reader(lib):
    gulp = 4096
    ring = Ring('blocking')
    _check(L.bfRingResize(ring.obj, gulp, 2 * gulp, 1))
    _check(L.bfRingBeginWriting(ring.obj))
    ring.begin_sequence('s', 1)
    reader = ring.open_earliest(guarantee=True)
    for _ in range(2):
        _check(L.bfRingSpanCommit(ring.reserve(gulp), gulp))
    # the ring is full of data the reader still holds: non-blocking says so ...
    with pytest.raises(IOError):
        ring.reserve(gulp, nonblocking=True)
    # ... and a blocking reservation waits until the reader moves on
    done = threading.Event()

    def blocked():
        _check(L.bfRingSpanCommit(ring.reserve(gulp), gulp))
        done.set()
    t = threading.Thread(target=blocked)
    t.start()
    assert not done.wait(0.3)
    span = ctypes.c_void_p()
    _check(L.bfRingSpanAcquire(ctypes.byref(span), reader, gulp, gulp))      # lets go of the first gulp
    assert done.wait(10)
    t.join()
    _check(L.bfRingSpanRelease(span))
    _check(L.bfRingSequenceClose(reader))
    ring.destroy()


def test_unguaranteed_reader_sees_what_was_overwritten(lib):
    gulp = 4096
    ring = Ring('lossy')
    _check(L.bfRingResize(ring.obj, gulp, 2 * gulp, 1))
    _check(L.bfRingBeginWriting(ring.obj))
    ring.begin_sequence('s', 1)
    _check(L.bfRingSpanCommit(ring.reserve(gulp), gulp))
    reader = ring.open_earliest(guarantee=False)
    span = ctypes.c_void_p()
    _check(L.bfRingSpanAcquire(ctypes.byref(span), reader, 0, gulp))
    assert _get(L.bfRingSpanGetSizeOverwritten, span) == 0
    _check(L.bfRingSpanCommit(ring.reserve(gulp), gulp))          # the ring is full now ...
    half = ring.reserve(gulp // 2)                                   # ... and this laps the reader by half a gulp
    assert _get(L.bfRingSpanGetSizeOverwritten, span) == gulp // 2
    _check(L.bfRingSpanCommit(half, gulp // 2))
    _check(L.bfRingSpanRelease(span))
    # asking again for the start of the sequence gives what is left of it
    _check(L.bfRingSpanAcquire(ctypes.byref(span), reader, 0, gulp))
    inf = ring.info(span)
    assert (inf.offset, inf.size) == (gulp // 2, gulp // 2)
    _check(L.bfRingSpanRelease(span))
    _check(L.bfRingSequenceClose(reader))
    ring.destroy()


def test_status_codes_of_misuse():
    ring = Ring('misuse')
    h = ctypes.c_void_p()
    assert L.bfRingSpanReserve(ctypes.byref(h), ring.obj, 16, 1) == _bf.BF_STATUS_INVALID_ARGUMENT   # > contiguous span (0)
    assert L.bfRingSpanReserve(ctypes.byref(h), ring.obj, 0, 1) == _bf.BF_STATUS_INVALID_STATE       # never sized
    _check(L.bfRingResize(ring.obj, 100, 400, 2))
    assert _get(L.bfRingGetName, ring.obj) == b'misuse'
    assert _get(L.bfRingGetSpace, ring.obj) == _bf.BF_SPACE_SYSTEM
    _check(L.bfRingLock(ring.obj))
    assert _get(L.bfRingLockedGetContiguousSpan, ring.obj) == 4096       # rounded up to the alignment
    assert _get(L.bfRingLockedGetTotalSpan, ring.obj) == 4096           # power of two >= alignment
    assert _get(L.bfRingLockedGetStride, ring.obj) == 8192
    assert _get(L.bfRingLockedGetNRinglet, ring.obj) == 2
    assert _get(L.bfRingLockedGetData, ring.obj) % 4096 == 0
    _check(L.bfRingUnlock(ring.obj))
    assert L.bfRingEndWriting(ring.obj) == _bf.BF_STATUS_INVALID_STATE       # before begin
    _check(L.bfRingBeginWriting(ring.obj))
    assert L.bfRingBeginWriting(ring.obj) == _bf.BF_STATUS_INVALID_STATE
    assert L.bfRingSpanReserve(ctypes.byref(h), ring.obj, 4097, 1) == _bf.BF_STATUS_INVALID_ARGUMENT
    assert L.bfRingSequenceBegin(ctypes.byref(h), ring.obj, b's', 1, 0, None, 3, 0) == _bf.BF_STATUS_INVALID_ARGUMENT
    assert L.bfRingSequenceBegin(ctypes.byref(h), ring.obj, b's', 1, 4, None, 1, 0) == _bf.BF_STATUS_INVALID_ARGUMENT
    seq = ring.begin_sequence('s', 1, b'abc', 2)
    assert L.bfRingSequenceBegin(ctypes.byref(h), ring.obj, b't', 2, 0, None, 1, 0) == _bf.BF_STATUS_INVALID_STATE
    assert L.bfRingSequenceOpen(ctypes.byref(h), ring.obj, b'nope', 1) == _bf.BF_STATUS_INVALID_ARGUMENT
    assert L.bfRingSequenceOpenAt(ctypes.byref(h), ring.obj, 0, 1) == _bf.BF_STATUS_INVALID_ARGUMENT
    assert L.bfRingSequenceOpenAt(ctypes.byref(h), ring.obj, 2 ** 64 - 1, 1) == _bf.BF_STATUS_INVALID_ARGUMENT
    w = ring.reserve(64)
    assert L.bfRingEndWriting(ring.obj) == _bf.BF_STATUS_INVALID_STATE       # a span is open
    assert L.bfRingSpanCommit(w, 65) == _bf.BF_STATUS_INVALID_ARGUMENT
    _check(L.bfRingSpanCommit(w, 64))
    _check(L.bfRingSequenceEnd(seq, 0))
    _check(L.bfRingEndWriting(ring.obj))
    assert _get(L.bfRingWritingEnded, ring.obj) == 1
    _check(L.bfRingSequenceOpen(ctypes.byref(h), ring.obj, b's', 0))
    span = ctypes.c_void_p()
    assert L.bfRingSpanAcquire(ctypes.byref(span), h, 64, 8) == _bf.BF_STATUS_END_OF_DATA
    _check(L.bfRingSpanAcquire(ctypes.byref(span), h, 60, 8))
    assert ring.info(span).size == 4                                           # cut at the end of the sequence
    _check(L.bfRingSpanRelease(span))
    assert L.bfRingSequenceNext(h) == _bf.BF_STATUS_END_OF_DATA
    _check(L.bfRingSequenceClose(h))
    for fn, args in ((L.bfRingDestroy, (None,)), (L.bfRingSpanRelease, (None,)), (L.bfRingSequenceClose, (None,)),
                     (L.bfRingResize, (None, 1, 1, 1))):
        assert fn(*args) == _bf.BF_STATUS_INVALID_HANDLE
    assert L.bfRingCreate(None, b'x', 1) == _bf.BF_STATUS_INVALID_POINTER
    assert L.bfRingCreate(ctypes.byref(h), b'x', 77) == _bf.BF_STATUS_INVALID_ARGUMENT
    ring.destroy()


def test_opening_on_an_ended_empty_ring_is_end_of_data(lib):
    ring = Ring('empty')
    _check(L.bfRingResize(ring.obj, 64, 256, 1))
    _check(L.bfRingBeginWriting(ring.obj))
    _check(L.bfRingEndWriting(ring.obj))
    h = ctypes.c_void_p()
    assert L.bfRingSequenceOpenEarliest(ctypes.byref(h), ring.obj, 1) == _bf.BF_STATUS_END_OF_DATA
    assert L.bfRingSequenceOpenLatest(ctypes.byref(h), ring.obj, 0) == _bf.BF_STATUS_END_OF_DATA
    # the failed guaranteed open left nothing pinned: the writer side would not block
    ring.destroy()


def test_ring_memory_placement_request_is_honoured_or_harmless():
    ring = Ring('numa')
    assert _get(L.bfRingGetAffinity, ring.obj) == -1
    _check(L.bfRingSetAffinity(ring.obj, 0))
    assert _get(L.bfRingGetAffinity, ring.obj) == 0
    assert L.bfRingSetAffinity(ring.obj, -2) == _bf.BF_STATUS_INVALID_ARGUMENT
    _check(L.bfRingResize(ring.obj, 1 << 16, 1 << 18, 1))       # allocates under the node preference
    w = ring.reserve(1 << 16)
    span_view(ring.info(w), 0)[:] = 5
    _check(L.bfRingSpanCommit(w, 1 << 16))
    ring.destroy()


def proclog_root():
    return os.path.join(os.environ['BIFROST_B200_PROCLOG_DIR'], str(os.getpid()))


def test_proclog_files():
    log = ctypes.c_void_p()
    _check(_bf.bfProcLogCreate(ctypes.byref(log), b'myblock/perf'))
    path = os.path.join(proclog_root(), 'myblock', 'perf')
    _check(_bf.bfProcLogUpdate(log, b'acquire_time : 0.5\nprocess_time : 1.5\n'))
    assert open(path).read() == 'acquire_time : 0.5\nprocess_time : 1.5\n'
    _check(_bf.bfProcLogUpdate(log, b'acquire_time : 0.25\n'))          # rewritten, not appended
    assert open(path).read() == 'acquire_time : 0.25\n'
    # a second log of the same name gets its block numbered (ref proclog.cpp:103-121)
    twin = ctypes.c_void_p()
    _check(_bf.bfProcLogCreate(ctypes.byref(twin), b'myblock/perf'))
    _check(_bf.bfProcLogUpdate(twin, b'x : 1\n'))
    assert open(os.path.join(proclog_root(), 'myblock_2', 'perf')).read() == 'x : 1\n'
    _check(_bf.bfProcLogDestroy(twin))
    _check(_bf.bfProcLogDestroy(log))
    assert not os.path.exists(path)
    assert _bf.bfProcLogCreate(None, b'a/b') == _bf.BF_STATUS_INVALID_POINTER
    assert _bf.bfProcLogUpdate(None, b'') == _bf.BF_STATUS_INVALID_HANDLE
    # every ring describes itself under rings/<name>
    ring = Ring('logged')
    _check(L.bfRingResize(ring.obj, 100, 1000, 3))
    text = open(os.path.join(proclog_root(), 'rings', 'logged')).read()
    fields = dict(line.split(':') for line in text.strip().splitlines())
    fields = {k.strip(): v.strip() for k, v in fields.items()}
    assert fields['space'] == 'system' and fields['nringlet'] == '3'
    assert int(fields['span']) == 4096 and int(fields['ghost']) == 4096 and int(fields['stride']) == 8192
    ring.destroy()
    assert not os.path.exists(os.path.join(proclog_root(), 'rings', 'logged'))


def test_thread_affinity():
    before = os.sched_getaffinity(0)
    result = {}

    def body():
        try:
            cores = sorted(os.sched_getaffinity(0))
            _check(_bf.bfAffinitySetCore(cores[-1]))
            result['bound'] = _get(_bf.bfAffinityGetCore)
            result['sched'] = os.sched_getaffinity(0)
            assert _bf.bfAffinitySetCore(10 ** 6) == _bf.BF_STATUS_INVALID_ARGUMENT
            _check(_bf.bfAffinitySetCore(-1))
            result['unbound'] = _get(_bf.bfAffinityGetCore)
            result['last'] = cores[-1]
            result['ncore'] = os.cpu_count()
        except Exception as e:      # pragma: no cover
            result['error'] = e
    t = threading.Thread(target=body)      # a thread of its own: the binding is per thread
    t.start()
    t.join()
    assert 'error' not in result, result['error']
    assert result['bound'] == result['last'] and result['sched'] == {result['last']}
    assert result['unbound'] == (-1 if result['ncore'] > 1 else 0)
    assert _bf.bfAffinitySetOpenMPCores(0, None) == _bf.BF_STATUS_UNSUPPORTED
    assert os.sched_getaffinity(0) == before


# --------------------------------------------------------------------------
# rings in device memory: ghost copies are device-to-device, on the caller's stream
# --------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.timeout(120)
def test_cuda_space_ring_round_trip():
    gulp, ngulp, nringlet = 3000, 40, 2
    ring = Ring('device', space='cuda')
    _check(L.bfRingResize(ring.obj, gulp, 4 * gulp, nringlet))
    assert _get(L.bfRingGetSpace, ring.obj) == _bf.BF_SPACE_CUDA
    _check(L.bfRingBeginWriting(ring.obj))
    seq = ring.begin_sequence('dev', 7, b'{}', nringlet)
    reader = ring.open_earliest(guarantee=True)
    for i in range(ngulp):
        w = ring.reserve(gulp)
        inf = ring.info(w)
        assert _get(_bf.bfGetSpace, inf.data) == _bf.BF_SPACE_CUDA
        src = np.stack([payload(i, r, gulp) for r in range(nringlet)])
        _check(_bf.bfMemcpy2D(inf.data, inf.stride, _bf.BF_SPACE_CUDA, src.ctypes.data, gulp, _bf.BF_SPACE_SYSTEM,
                              gulp, nringlet))
        _check(_bf.bfStreamSynchronize())
        _check(L.bfRingSpanCommit(w, gulp))
        # read it back half a gulp late, so that read spans straddle the write
        # spans and both kinds of ghost copy (write ran over the end / read
        # runs over the end) happen on the device
        if i >= 1:
            span = ctypes.c_void_p()
            _check(L.bfRingSpanAcquire(ctypes.byref(span), reader, (i - 1) * gulp + gulp // 2, gulp))
            rinf = ring.info(span)
            assert rinf.size == gulp
            got = np.zeros((nringlet, gulp), np.uint8)
            _check(_bf.bfMemcpy2D(got.ctypes.data, gulp, _bf.BF_SPACE_SYSTEM, rinf.data, rinf.stride, _bf.BF_SPACE_CUDA,
                                  gulp, nringlet))
            _check(_bf.bfStreamSynchronize())
            for r in range(nringlet):
                want = np.concatenate([payload(i - 1, r, gulp)[gulp // 2:], payload(i, r, gulp)[:gulp // 2]])
                np.testing.assert_array_equal(got[r], want)
            _check(L.bfRingSpanRelease(span))
    # growing a device ring keeps its contents
    _check(L.bfRingResize(ring.obj, 2 * gulp, 16 * gulp, nringlet))
    span = ctypes.c_void_p()
    _check(L.bfRingSpanAcquire(ctypes.byref(span), reader, (ngulp - 2) * gulp, 2 * gulp))
    rinf = ring.info(span)
    got = np.zeros((nringlet, 2 * gulp), np.uint8)
    _check(_bf.bfMemcpy2D(got.ctypes.data, 2 * gulp, _bf.BF_SPACE_SYSTEM, rinf.data, rinf.stride, _bf.BF_SPACE_CUDA,
                          2 * gulp, nringlet))
    _check(_bf.bfStreamSynchronize())
    for r in range(nringlet):
        np.testing.assert_array_equal(got[r], np.concatenate([payload(ngulp - 2, r, gulp), payload(ngulp - 1, r, gulp)]))
    _check(L.bfRingSpanRelease(span))
    _check(L.bfRingSequenceEnd(seq, 0))
    _check(L.bfRingSequenceClose(reader))
    _check(L.bfRingEndWriting(ring.obj))
    ring.destroy()
