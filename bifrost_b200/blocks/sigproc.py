"""Sigproc source and sink blocks (mirror python/bifrost/blocks/sigproc.py:51-390):
read_sigproc emits [time, pol, freq] from filterbank / time-series files;
write_sigproc writes filterbanks ([time, pol, freq], optionally one file per
beam) and time series ([time, pol], or one .tim per trial for
[dispersion, time, pol] -- the FDMT block's output)."""
import os

import numpy as np

from bifrost_b200.pipeline import SourceBlock, SinkBlock
from bifrost_b200.DataType import DataType
from bifrost_b200.units import convert_units
from bifrost_b200 import sigproc


def _mjd2unix(mjd):
    return (mjd - 40587) * 86400


def _unix2mjd(unix):
    return unix / 86400. + 40587


def _copy_item_if_exists(dst, src, key, newkey=None):
    if key in src:
        dst[key if newkey is None else newkey] = src[key]


class SigprocSourceBlock(SourceBlock):
    def __init__(self, filenames, gulp_nframe, unpack=True, *args, **kwargs):
        super(SigprocSourceBlock, self).__init__(filenames, gulp_nframe, *args, **kwargs)
        self.unpack = unpack

    def create_reader(self, sourcename):
        return sigproc.SigprocFile(sourcename)

    # sigproc keyword -> (output header key, default)
    _PASSTHROUGH = (('source_name', 'source_name', None), ('rawdatafile', 'rawdatafile', None),
                    ('az_start', 'az_start', None), ('za_start', 'za_start', None),
                    ('src_raj', 'raj', None), ('src_dej', 'dej', None), ('refdm', 'refdm', 0.),
                    ('ibeam', 'ibeam', None), ('nbeams', 'nbeams', None))

    def on_sequence(self, ireader, sourcename):
        sp = ireader.header
        if sp['data_type'] not in (1, 2, 6):        # filterbank, time series, dedispersed subbands
            raise ValueError("Unsupported sigproc data_type %r" % sp['data_type'])
        frames = [f for f in ('pulsarcentric', 'barycentric') if sp.get(f, 0)]
        t0 = _mjd2unix(sp['tstart'])
        nbit = sp['nbits']
        # 32-bit sigproc samples are floats (the reference labels them u32/i32)
        sample_type = 'f32' if nbit == 32 else '%s%d' % ('i' if ireader.signed else 'u', nbit)
        tensor = dict(dtype=sample_type, shape=[-1, sp.get('nifs', 1), sp['nchans']],
                      labels=['time', 'pol', 'freq'],
                      scales=[(t0, sp['tsamp']), None, (sp.get('fch1', 0.), sp.get('foff', 0.))],
                      units=['s', None, 'MHz'])
        ohdr = {'_tensor': tensor, 'frame_rate': 1. / sp['tsamp'], 'refdm_units': 'pc cm^-3',
                'telescope': sigproc.id2telescope(sp.get('telescope_id')),
                'machine': sigproc.id2machine(sp.get('machine_id')),
                'coord_frame': frames[0] if frames else 'topocentric',
                'time_tag': int(round(t0 * 2 ** 32)), 'name': sourcename}
        for key, okey, default in self._PASSTHROUGH:
            ohdr[okey] = sp.get(key, default)
        return [ohdr]

    def on_data(self, reader, ospans):
        ospan = ospans[0]
        nbyte = reader.readinto(ospan.data)
        return [nbyte // reader.frame_nbyte]


def read_sigproc(filenames, gulp_nframe, unpack=True, *args, **kwargs):
    """Read SIGPROC files.  Output: ['time', 'pol', 'freq'], u/i8, u/i16 or f32, system space."""
    return SigprocSourceBlock(filenames, gulp_nframe, unpack, *args, **kwargs)


class SigprocSinkBlock(SinkBlock):
    def __init__(self, iring, path=None, *args, **kwargs):
        super(SigprocSinkBlock, self).__init__(iring, *args, **kwargs)
        self.path = path or ''

    def define_valid_input_spaces(self):
        return ('system',)

    def on_sequence(self, iseq):
        ihdr = iseq.header
        itensor = ihdr['_tensor']
        axnames, shape = list(itensor['labels']), list(itensor['shape'])
        scales, units = list(itensor['scales']), list(itensor['units'])
        ndim = len(shape)
        dtype = DataType(itensor['dtype'])
        hdr = {}
        for key in ('source_name', 'rawdatafile', 'az_start', 'za_start'):
            _copy_item_if_exists(hdr, ihdr, key)
        if hdr.get('rawdatafile') is not None:
            # the file's name, as for the output file below: a source block's full
            # path can be longer than the 79 bytes a sigproc header string holds
            hdr['rawdatafile'] = os.path.basename(str(hdr['rawdatafile']))
        _copy_item_if_exists(hdr, ihdr, 'raj', 'src_raj')
        _copy_item_if_exists(hdr, ihdr, 'dej', 'src_dej')
        if ihdr.get('telescope') is not None:
            hdr['telescope_id'] = sigproc.telescope2id(ihdr['telescope'])
        if ihdr.get('machine') is not None:
            hdr['machine_id'] = sigproc.machine2id(ihdr['machine'])
        for key in ('telescope_id', 'machine_id', 'ibeam', 'nbeams'):
            _copy_item_if_exists(hdr, ihdr, key)
        hdr['nbits'] = dtype.itemsize_bits
        if dtype.is_integer and dtype.is_signed:
            hdr['signed'] = True
        coord_frame = ihdr.get('coord_frame')
        hdr['pulsarcentric'] = (coord_frame == 'pulsarcentric')
        hdr['barycentric'] = (coord_frame == 'barycentric')
        filename = os.path.join(self.path, os.path.basename(str(ihdr['name'])))
        self.ofile, self.ofiles = None, None

        def refdm():
            if ihdr.get('refdm') is not None:
                hdr['refdm'] = convert_units(ihdr['refdm'], ihdr.get('refdm_units', 'pc cm^-3'), 'pc cm^-3')

        if ndim >= 3 and axnames[-3:] == ['time', 'pol', 'freq']:
            self.data_format = 'filterbank'
            assert dtype.is_real
            hdr['data_type'] = 1
            hdr['nifs'], hdr['nchans'] = shape[-2], shape[-1]
            hdr['tstart'] = _unix2mjd(scales[-3][0])
            hdr['tsamp'] = convert_units(scales[-3][1], units[-3], 's')
            hdr['fch1'] = convert_units(scales[-1][0], units[-1], 'MHz')
            hdr['foff'] = convert_units(scales[-1][1], units[-1], 'MHz')
            refdm()
            if ndim == 3:
                self.ofile = open(filename + '.fil', 'wb')
                sigproc.write_header(hdr, self.ofile)
            elif ndim == 4:
                if axnames[-4] != 'beam':
                    raise ValueError("Expected first axis to be 'beam' got '%s'" % axnames[-4])
                nbeam = shape[-4]
                hdr['nbeams'] = nbeam
                self.ofiles = [open(filename + '.%06iof.%06i.fil' % (b + 1, nbeam), 'wb') for b in range(nbeam)]
                for b in range(nbeam):
                    hdr['ibeam'] = b
                    sigproc.write_header(hdr, self.ofiles[b])
            else:
                raise ValueError("Too many dimensions")
        elif ndim >= 2 and 'time' in axnames and 'pol' in axnames:
            pol_axis = axnames.index('pol')
            if pol_axis != ndim - 1:
                for lst in (axnames, shape, scales, units):
                    lst.append(lst.pop(pol_axis))
            self.pol_axis = pol_axis
            self.data_format = 'timeseries'
            assert dtype.is_real
            hdr['data_type'] = 2
            hdr['nchans'] = 1
            hdr['nifs'] = shape[-1]
            hdr['tstart'] = _unix2mjd(scales[-2][0])
            hdr['tsamp'] = convert_units(scales[-2][1], units[-2], 's')
            if 'cfreq' in ihdr and 'bw' in ihdr:
                hdr['fch1'] = convert_units(ihdr['cfreq'], ihdr['cfreq_units'], 'MHz')
                hdr['foff'] = convert_units(ihdr['bw'], ihdr['bw_units'], 'MHz')
            if ndim == 2:
                refdm()
                self.ofile = open(filename + '.tim', 'wb')
                sigproc.write_header(hdr, self.ofile)
            elif ndim == 3:
                if axnames[-3] != 'dispersion':
                    raise ValueError("Expected first axis to be 'dispersion' got '%s'" % axnames[-3])
                dm0, ddm = scales[-3]
                dms = [convert_units(dm0 + ddm * d, units[-3], 'pc cm^-3') for d in range(shape[-3])]
                self.ofiles = [open(filename + '.%09.2f.tim' % dm, 'wb') for dm in dms]
                for d, dm in enumerate(dms):
                    hdr['refdm'] = dm
                    sigproc.write_header(hdr, self.ofiles[d])
            else:
                raise ValueError("Too many dimensions")
        else:
            raise ValueError("Axis labels do not correspond to a known data format: " + str(axnames) +
                             "\nKnown formats are:\n  [time, pol, freq]\n  [beam, time, pol, freq]\n"
                             "  [time, pol]\n  [dispersion, time, pol]")

    def on_sequence_end(self, iseq):
        if self.ofile is not None:
            self.ofile.close()
        for f in self.ofiles or []:
            f.close()

    def on_data(self, ispan):
        idata = np.asarray(ispan.data)
        if self.data_format == 'timeseries' and self.pol_axis != idata.ndim - 1:
            perm = list(range(idata.ndim))
            perm.append(perm.pop(self.pol_axis))
            idata = np.ascontiguousarray(idata.transpose(perm))
        if self.ofile is not None:
            idata.tofile(self.ofile)
        else:
            # the leading axis (beam / dispersion) is not the frame axis: one file each
            for k in range(idata.shape[0]):
                np.ascontiguousarray(idata[k]).tofile(self.ofiles[k])


def write_sigproc(iring, path=None, *args, **kwargs):
    """Write [time, pol, freq] (+beam) filterbanks or [time, pol] (+dispersion) time series."""
    return SigprocSinkBlock(iring, path, *args, **kwargs)
