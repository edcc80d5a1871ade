"""Sigproc headers and files (mirrors python/bifrost/sigproc2.py:64-260 and the
parts of sigproc.py the blocks use): the keyword/value header between
HEADER_START and HEADER_END (int32 length-prefixed strings, '=i' / '=d' / '=b'
values) followed by raw samples [time][if][chan]."""
import struct
import warnings

import numpy as np

_string_values = ['source_name', 'rawdatafile']
_double_values = ['az_start', 'za_start', 'src_raj', 'src_dej', 'tstart', 'tsamp', 'period',
                  'fch1', 'foff', 'refdm']
_integer_values = ['nchans', 'telescope_id', 'machine_id', 'data_type', 'ibeam', 'nbeams', 'nbits',
                   'barycentric', 'pulsarcentric', 'nbins', 'nsamples', 'nifs', 'npuls']
_character_values = ['signed']

_telescopes = {0: 'Fake', 1: 'Arecibo', 2: 'Ooty', 3: 'Nancay', 4: 'Parkes', 5: 'Jodrell', 6: 'GBT',
               7: 'GMRT', 8: 'Effelsberg', 9: 'Effelsberg LOFAR', 10: 'UTR-2', 11: 'LOFAR', 12: 'MWA',
               20: 'CHIME', 52: 'LWA-OV', 53: 'LWA-SV', 64: 'MeerKAT', 65: 'KAT-7', 82: 'eMerlin'}
_machines = {0: 'FAKE', 1: 'PSPM', 2: 'WAPP', 3: 'AOFTM', 4: 'BPP', 5: 'OOTY', 6: 'SCAMP', 7: 'GMRTFB',
             8: 'PULSAR2000', 9: 'UNKNOWN', 11: 'BG/P', 12: 'PDEV', 20: 'GUPPI', 52: 'LWA-DP',
             53: 'LWA-ADP'}


def id2telescope(id_):
    return _telescopes.get(id_, 'unknown')


def telescope2id(name):
    """Name -> id; 'unknown' (what id2telescope gives a file without the card)
    maps back to None so that write_header leaves the card out again, as the
    reference's defaultdict round trip does (sigproc2.py:106-149)."""
    for k, v in _telescopes.items():
        if v == name:
            return k
    if name == 'unknown':
        return None
    raise ValueError("Unknown telescope: %r" % name)


def id2machine(id_):
    return _machines.get(id_, 'unknown')


def machine2id(name):
    for k, v in _machines.items():
        if v == name:
            return k
    if name == 'unknown':
        return None
    raise ValueError("Unknown machine: %r" % name)


def _write_string(f, text):
    f.write(struct.pack('=i', len(text)))
    f.write(text.encode())


def write_header(hdr, f):
    """Keys with value None are skipped; unknown keys warn (sigproc2.py:180-199).
    A string value of 80 bytes or more is an error: no sigproc reader (this
    one, the reference's, SIGPROC's 80-character fields) can read it back."""
    _write_string(f, "HEADER_START")
    for key, val in hdr.items():
        if val is None:
            continue
        if key in _string_values:
            if len(val.encode()) >= 80:
                raise ValueError("sigproc header %s is %d bytes; readers take at most 79: %r"
                                 % (key, len(val.encode()), val))
            _write_string(f, key)
            _write_string(f, val)
        elif key in _double_values:
            _write_string(f, key)
            f.write(struct.pack('=d', float(val)))
        elif key in _integer_values:
            _write_string(f, key)
            f.write(struct.pack('=i', int(val)))
        elif key in _character_values:
            _write_string(f, key)
            f.write(struct.pack('=b', int(val)))
        else:
            warnings.warn("Unknown sigproc header key: '%s'" % key, RuntimeWarning)
    _write_string(f, "HEADER_END")


def _read_string(f):
    raw = f.read(4)
    if len(raw) < 4:
        return None
    length = struct.unpack('=i', raw)[0]
    if length < 0 or length >= 80:
        return None
    return f.read(length).decode()


def read_header(f):
    if _read_string(f) != "HEADER_START":
        raise ValueError("Missing HEADER_START")
    expecting, header = None, {}
    while True:
        key = _read_string(f)
        if key is None:
            raise ValueError("Failed to parse header")
        if key == 'HEADER_END':
            break
        if key in _string_values:
            expecting = key
        elif key in _double_values:
            header[key] = struct.unpack('=d', f.read(8))[0]
        elif key in _integer_values:
            header[key] = struct.unpack('=i', f.read(4))[0]
        elif key in _character_values:
            header[key] = struct.unpack('=b', f.read(1))[0]
        elif expecting is not None:
            header[expecting] = key
            expecting = None
        else:
            warnings.warn("Unknown header key: '%s'" % key, RuntimeWarning)
    header.setdefault('nchans', 1)
    header['header_size'] = f.tell()
    return header


class SigprocFile(object):
    """Streaming reader of filterbank / time-series files (8-, 16-, 32-bit
    samples; packed sub-byte files are rejected here -- unpack them on the
    device with bf.blocks.unpack)."""

    def __init__(self, filename=None):
        self.f = None
        if filename is not None:
            self.open(filename)

    def open(self, filename):
        self.f = open(filename, 'rb')
        self.header = read_header(self.f)
        self.header_size = self.header['header_size']
        self.nbit = self.header['nbits']
        self.signed = bool(self.header.get('signed', 0))
        self.nifs = self.header.get('nifs', 1)
        self.nchans = self.header['nchans']
        if self.nbit not in (8, 16, 32):
            raise ValueError("nbits = %d needs the device unpacker" % self.nbit)
        if self.nbit == 32:
            self.dtype = np.dtype(np.float32)
        else:
            self.dtype = np.dtype(('i' if self.signed else 'u') + str(self.nbit // 8))
        self.frame_shape = (self.nifs, self.nchans)
        self.frame_nbyte = self.nifs * self.nchans * self.dtype.itemsize
        return self

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
        return False

    def close(self):
        if self.f is not None:
            self.f.close()
            self.f = None

    def readinto(self, buf):
        """Reads whole frames into the writable array `buf`; returns bytes read."""
        view = np.asarray(buf).reshape(-1).view(np.uint8)
        nbyte = self.f.readinto(view)
        return nbyte - nbyte % self.frame_nbyte
