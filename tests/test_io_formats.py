"""File formats either side of the hot path (SURVEY 8f.4): GUPPI RAW block
headers and the source block, sigproc headers and the source / sink blocks.
Golden bytes and parsed headers come from the reference's own Python
(tests/golden/make_io_golden.py ran python/bifrost/sigproc2.py and guppi_raw.py)."""
import base64
import io
import json
import os
import sys
from copy import deepcopy

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bifrost_b200 as bf  # noqa: E402
from bifrost_b200 import blocks, guppi_raw, sigproc  # noqa: E402
from bifrost_b200.pipeline import Pipeline  # noqa: E402

GOLD = json.load(open(os.path.join(ROOT, 'tests', 'golden', 'io_golden.json')))


@pytest.mark.parametrize("name", sorted(GOLD['sigproc']))
def test_sigproc_header_bytes_match_the_reference_writer(name):
    g = GOLD['sigproc'][name]
    f = io.BytesIO()
    sigproc.write_header(dict((k, v) for k, v in g['header']), f)
    assert f.getvalue() == base64.b64decode(g['bytes'])
    assert sigproc.read_header(io.BytesIO(f.getvalue())) == g['parsed']


def test_guppi_header_matches_the_reference_reader():
    g = GOLD['guppi']
    f = io.BytesIO(base64.b64decode(g['bytes']) + b'\x01\x02\x03\x04')
    assert guppi_raw.read_header(f) == g['parsed']
    assert f.tell() == g['data_offset']
    assert f.read(4) == b'\x01\x02\x03\x04'


class Collect(object):
    def __init__(self):
        self.chunks, self.headers = [], []

    def seq(self, iseq):
        self.headers.append(deepcopy(iseq.header))

    def data(self, ispan):
        self.chunks.append(np.array(np.asarray(ispan.data)))


def guppi_file(path, nblock, nchan, ntime, directio):
    rng = np.random.default_rng(2)
    data = rng.integers(-128, 128, size=(nblock, nchan, ntime, 2, 2), dtype=np.int8)
    with open(path, 'wb') as f:
        for b in range(nblock):
            hdr = dict(BACKEND='GUPPI', TELESCOP='GBT', SRC_NAME='FAKE', OBSFREQ=1500.0, OBSBW=-187.5,
                       OBSNCHAN=nchan, NPOL=4, NBITS=8, BLOCSIZE=nchan * ntime * 4, PKTIDX=b * 16,
                       PKTSIZE=8192, STT_IMJD=58849, STT_SMJD=43200, RA=53.2475, DEC=54.5787, CHAN_DM=0.0)
            if directio:
                hdr['DIRECTIO'] = 1
            guppi_raw.write_header(hdr, f)
            data[b].tofile(f)
    return data


@pytest.mark.parametrize("directio", [False, True])
@pytest.mark.parametrize("gulp", [1, 2])
def test_guppi_source_block(tmp_path, directio, gulp):
    path = str(tmp_path / 'fake.raw')
    nblock, nchan, ntime = 5, 8, 64
    data = guppi_file(path, nblock, nchan, ntime, directio)
    out = Collect()
    with Pipeline() as p:
        src = blocks.read_guppi_raw([path], gulp_nframe=gulp)
        blocks.callback_sink(src, out.seq, out.data)
        p.run()
    hdr = out.headers[0]
    t = hdr['_tensor']
    assert t['dtype'] == 'ci8' and t['shape'] == [-1, nchan, ntime, 2]
    assert t['labels'] == ['time', 'freq', 'fine_time', 'pol']
    df = -187.5 / nchan
    assert t['scales'][1] == pytest.approx((1500.0 - 0.5 * (nchan - 1) * df, df))
    assert t['scales'][2][1] == pytest.approx(1. / df / 1e6)
    assert hdr['telescope'] == 'GBT' and hdr['machine'] == 'GUPPI'
    got = np.concatenate(out.chunks, 0)
    got = np.stack([got['re'], got['im']], -1)
    np.testing.assert_array_equal(got, data)


def fil_header(nchan, npol, dtype):
    return {'_tensor': {'dtype': dtype, 'shape': [-1, npol, nchan], 'labels': ['time', 'pol', 'freq'],
                        'scales': [[1500000000.0, 1e-3], None, [1500.0, -0.5]], 'units': ['s', None, 'MHz']},
            'name': 'obs', 'gulp_nframe': 16, 'source_name': 'FAKE', 'telescope': 'GBT', 'machine': 'GUPPI',
            'coord_frame': 'topocentric', 'refdm': 0.0, 'refdm_units': 'pc cm^-3',
            # a source block's full path, longer than a sigproc header string holds
            'rawdatafile': '/data/' + 'd' * 100 + '/obs.raw'}


@pytest.mark.parametrize("dtype,npdt", [('f32', np.float32), ('i8', np.int8), ('u8', np.uint8)])
def test_sigproc_filterbank_round_trip(tmp_path, dtype, npdt):
    rng = np.random.default_rng(3)
    x = (rng.normal(size=(100, 2, 32)) * 20).astype(npdt)
    with Pipeline() as p:
        src = blocks.array_source(x, fil_header(32, 2, dtype), gulp_nframe=16)
        blocks.write_sigproc(src, path=str(tmp_path))
        p.run()
    path = str(tmp_path / 'obs.fil')
    with open(path, 'rb') as f:
        h = sigproc.read_header(f)
        body = np.fromfile(f, dtype=npdt)
    assert h['data_type'] == 1 and h['nifs'] == 2 and h['nchans'] == 32 and h['nbits'] == 8 * x.itemsize
    assert h['tstart'] == pytest.approx(1500000000.0 / 86400. + 40587) and h['tsamp'] == 1e-3
    assert (h['fch1'], h['foff']) == (1500.0, -0.5) and h['telescope_id'] == 6 and h['machine_id'] == 20
    assert h.get('signed', 0) == (1 if dtype == 'i8' else 0)
    assert h['rawdatafile'] == 'obs.raw'
    np.testing.assert_array_equal(body.reshape(x.shape), x)
    out = Collect()
    with Pipeline() as p:
        src = blocks.read_sigproc([path], gulp_nframe=32)
        blocks.callback_sink(src, out.seq, out.data)
        p.run()
    t = out.headers[0]['_tensor']
    assert t['dtype'] == dtype and t['shape'] == [-1, 2, 32] and t['labels'] == ['time', 'pol', 'freq']
    assert out.headers[0]['telescope'] == 'GBT'
    np.testing.assert_array_equal(np.concatenate(out.chunks, 0), x)


def test_sigproc_header_string_a_reader_cannot_take_is_an_error():
    """Strings of 80 bytes or more would make a file no sigproc reader parses."""
    sigproc.write_header(dict(source_name='x' * 79), io.BytesIO())
    with pytest.raises(ValueError):
        sigproc.write_header(dict(source_name='x' * 80), io.BytesIO())


def test_sigproc_file_without_id_cards_round_trips(tmp_path):
    """read_sigproc -> write_sigproc of a file that has no telescope_id / machine_id
    card: the ids come back as 'unknown' and the sink leaves the cards out again
    (the reference's defaultdict round trip, sigproc2.py:106-154)."""
    x = (np.arange(40 * 8).reshape(40, 1, 8) % 100).astype(np.uint8)
    src_path = str(tmp_path / 'noid.fil')
    with open(src_path, 'wb') as f:
        sigproc.write_header(dict(data_type=1, nchans=8, nifs=1, nbits=8, tstart=58000.0, tsamp=1e-3,
                                  fch1=1500.0, foff=-0.5, source_name='X'), f)
        x.tofile(f)
    outdir = tmp_path / 'out'
    outdir.mkdir()
    with Pipeline() as p:
        src = blocks.read_sigproc([src_path], gulp_nframe=16)
        blocks.write_sigproc(src, path=str(outdir))
        p.run()
    written = sorted(os.listdir(str(outdir)))
    assert len(written) == 1 and written[0].startswith('noid')
    with open(str(outdir / written[0]), 'rb') as f:
        h = sigproc.read_header(f)
        body = np.fromfile(f, dtype=np.uint8)
    assert 'telescope_id' not in h and 'machine_id' not in h
    assert h['nchans'] == 8 and h['source_name'] == 'X'
    np.testing.assert_array_equal(body.reshape(x.shape), x)
    assert sigproc.telescope2id('unknown') is None and sigproc.machine2id('unknown') is None
    with pytest.raises(ValueError):
        sigproc.telescope2id('Atlantis')


def test_sigproc_dispersion_trials_one_tim_per_dm(tmp_path):
    """[dispersion, time, pol] -- the FDMT block's output -- becomes one time series per trial."""
    rng = np.random.default_rng(4)
    ndm, ntime = 3, 50
    x = rng.normal(size=(ndm, ntime, 1)).astype(np.float32)
    hdr = {'_tensor': {'dtype': 'f32', 'shape': [ndm, -1, 1], 'labels': ['dispersion', 'time', 'pol'],
                       'scales': [[10.0, 2.5], [1500000000.0, 256e-6], None], 'units': ['pc cm^-3', 's', None]},
           'name': 'ddm', 'gulp_nframe': 20, 'cfreq': 1400.0, 'cfreq_units': 'MHz', 'bw': 400.0, 'bw_units': 'MHz'}
    with Pipeline() as p:
        src = blocks.array_source(x, hdr, gulp_nframe=20, frame_axis=1)
        blocks.write_sigproc(src, path=str(tmp_path))
        p.run()
    for d in range(ndm):
        dm = 10.0 + 2.5 * d
        with open(str(tmp_path / ('ddm.%09.2f.tim' % dm)), 'rb') as f:
            h = sigproc.read_header(f)
            body = np.fromfile(f, dtype=np.float32)
        assert h['data_type'] == 2 and h['refdm'] == dm and h['nchans'] == 1 and h['nifs'] == 1
        assert h['fch1'] == 1400.0 and h['foff'] == 400.0 and h['tsamp'] == 256e-6
        np.testing.assert_array_equal(body, x[d, :, 0])


def test_guppi_truncated_header_is_an_error_and_clean_eof_is_not(tmp_path):
    """A file that stops between blocks ends the sequence; one that stops inside
    a header is corrupt (the advisor's round-1 finding); NTIME must agree with
    BLOCSIZE."""
    import io
    import pytest
    from bifrost_b200 import guppi_raw
    hdr = {'OBSNCHAN': 2, 'NPOL': 4, 'NBITS': 8, 'BLOCSIZE': 2 * 4 * 2 * 2, 'OBSBW': 2.0, 'OBSFREQ': 100.0}
    f = io.BytesIO()
    guppi_raw.write_header(hdr, f)
    whole = f.getvalue()
    h = guppi_raw.read_header(io.BytesIO(whole))
    assert h.nbyte == len(whole) and h['NTIME'] == 4
    with pytest.raises(guppi_raw.EndOfFile):
        guppi_raw.read_header(io.BytesIO(b''))
    with pytest.raises(IOError) as e:
        guppi_raw.read_header(io.BytesIO(whole[:len(whole) - 100]))
    assert not isinstance(e.value, guppi_raw.EndOfFile)
