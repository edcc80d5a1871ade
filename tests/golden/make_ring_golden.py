"""Generates tests/golden/ring_traces.json.gz: random scripts of bfRing* calls
and what the REFERENCE's own ring answered to each of them (status codes, span
sizes / offsets / strides, geometry, sequence headers, CRCs of the bytes read).

The reference ring is oracle/_ref/libbifrost_ref_ring.so, compiled from the
unmodified src/{ring,ring_impl,proclog,fileutils,affinity,memory,common,cuda,
hw_locality}.cpp of the reference by oracle/ref_ring_build.sh (CPU only).
tests/test_ring.py replays the scripts on libbifrost_b200.so and compares
call by call; it does not need the reference tree.  `cases` are the short
scripts, `differential` the longer ones of the differential test.

    REF=<reference checkout> bash oracle/ref_ring_build.sh && python tests/golden/make_ring_golden.py
"""
import gzip
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import ringtrace  # noqa: E402

SEEDS = [(11, 260), (12, 260), (13, 260), (14, 260), (15, 260), (16, 260)]
DIFFERENTIAL_SEEDS = [(seed, 350) for seed in range(100, 112)]


def main():
    ref = ringtrace.load_reference()
    assert ref is not None, 'build oracle/_ref/libbifrost_ref_ring.so first (oracle/ref_ring_build.sh)'
    sets = {}
    for key, seeds in (('cases', SEEDS), ('differential', DIFFERENTIAL_SEEDS)):
        sets[key] = []
        for seed, nstep in seeds:
            script, trace = ringtrace.generate(ref, seed, nstep)
            sets[key].append(dict(seed=seed, script=script, trace=trace))
            print(key, seed, len(script), 'calls')
    out = os.path.join(HERE, 'ring_traces.json.gz')
    with gzip.GzipFile(out, 'wb', mtime=0) as f:
        f.write(json.dumps(dict(source='reference src/ring_impl.cpp via oracle/ref_ring_build.sh',
                                **sets), separators=(',', ':')).encode())
    print('wrote', out, os.path.getsize(out), 'bytes')


if __name__ == '__main__':
    main()
