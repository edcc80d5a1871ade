"""Generates tests/golden/io_golden.json from the REFERENCE's own Python
(python/bifrost/sigproc2.py write_header / _read_header, guppi_raw.py
read_header), executed from the reference checkout ($BIFROST_REFERENCE, by default
/root/reference) with its `bifrost.telemetry` import stubbed out (the package
itself cannot be imported without libbifrost).  The tests read the committed JSON."""
import base64
import io
import json
import os
import sys
import types

REF = os.path.join(os.environ.get('BIFROST_REFERENCE', '/root/reference'), 'python', 'bifrost')
HERE = os.path.dirname(os.path.abspath(__file__))


def load(name):
    pkg = types.ModuleType('bifrost')
    pkg.telemetry = types.SimpleNamespace(track_module=lambda: None)
    sys.modules['bifrost'] = pkg
    sys.modules['bifrost.telemetry'] = pkg.telemetry
    mod = types.ModuleType('ref_' + name)
    src = open(os.path.join(REF, name + '.py')).read()
    exec(compile(src, name + '.py', 'exec'), mod.__dict__)
    return mod


def main():
    sp = load('sigproc2')
    gr = load('guppi_raw')
    out = {}
    # ---- sigproc headers written by the reference
    hdrs = {
        'filterbank': dict(source_name='J0000+0000', rawdatafile='synthetic.raw', az_start=12.5, za_start=30.25,
                           src_raj=123456.7, src_dej=-12345.6, telescope_id=6, machine_id=20, nbits=32,
                           pulsarcentric=False, barycentric=False, data_type=1, nifs=2, nchans=64,
                           tstart=58000.125, tsamp=1.024e-3, fch1=1500.0, foff=-0.5, refdm=None),
        'timeseries_i8': dict(nbits=8, signed=True, pulsarcentric=False, barycentric=True, data_type=2,
                              nchans=1, nifs=1, tstart=59000.5, tsamp=256e-6, refdm=56.75),
    }
    out['sigproc'] = {}
    for name, h in hdrs.items():
        f = io.BytesIO()
        sp.write_header(h, f)
        raw = f.getvalue()
        back = sp._read_header(io.BytesIO(raw))
        out['sigproc'][name] = dict(header=list(h.items()), bytes=base64.b64encode(raw).decode(), parsed=back)
    # ---- GUPPI headers parsed by the reference
    cards = [
        "BACKEND = 'GUPPI   '", "TELESCOP= 'GBT     '", "SRC_NAME= 'B0329+54'", "OBSFREQ = 1500.0",
        "OBSBW   = -187.5", "OBSNCHAN= 64", "NPOL    = 4", "NBITS   = 8", "BLOCSIZE= 131072",
        "PKTIDX  = 1024", "PKTSIZE = 8192", "STT_IMJD= 58849", "STT_SMJD= 43200", "TBIN    = 3.41333e-07",
        "RA      = 53.2475", "DEC     = 54.5787", "AZ      = 100.5", "ZA      = 20.25", "CHAN_DM = 26.7641",
        "DIRECTIO= 1",
    ]
    raw = b''.join(c.ljust(80).encode() for c in cards) + 'END'.ljust(80).encode()
    raw += b' ' * (512 - len(raw) % 512)
    f = io.BytesIO(raw + b'\x01\x02\x03\x04')
    parsed = gr.read_header(f)
    out['guppi'] = dict(bytes=base64.b64encode(raw).decode(), parsed=parsed, data_offset=f.tell())
    json.dump(out, open(os.path.join(HERE, 'io_golden.json'), 'w'), indent=1, sort_keys=True)
    print('wrote io_golden.json')


if __name__ == '__main__':
    main()
