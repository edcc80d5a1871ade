"""Compact stand-ins for reference outputs too large to store whole.

An output that must match bit for bit keeps the SHA-256 of its bits and a
small sample that shows where a mismatch is.  All NaNs hash alike, as the
comparisons treat any two NaNs as equal.  An output compared within a
tolerance keeps a larger sample plus, for every BLOCK consecutive values, their
sum and the sum of their magnitudes: a value outside the sample that is off
by more than the tolerance allows still moves its block's sum out of bounds.
An output of at most SAMPLE values is stored whole and compared value for
value, with neither."""
import hashlib

import numpy as np

SAMPLE_EXACT = 512      # beside a digest, the sample only locates a mismatch
SAMPLE = 4096           # values of an output compared within a tolerance
BLOCK = 64              # values per stored block sum


def sha256(a):
    a = np.ascontiguousarray(a)
    if a.dtype.kind in 'fc':
        a = np.where(np.isnan(a), np.array(np.nan, a.dtype), a)
    return hashlib.sha256(a.tobytes()).hexdigest()


def block_sums(a):
    """(sum, sum of magnitudes) of every BLOCK consecutive values of `a`, in
    float64 / complex128; the last block is padded with zeros."""
    v = np.asarray(a).reshape(-1)
    v = np.concatenate([v, np.zeros((-v.size) % BLOCK, v.dtype)]).reshape(-1, BLOCK)
    wide = np.complex128 if v.dtype.kind == 'c' else np.float64
    return v.astype(wide).sum(1), np.abs(v.astype(wide)).sum(1)


def pack(key, a, exact, seed=0):
    """The entries of `a` to store under `key` in an .npz file."""
    a = np.asarray(a)
    whole = a.size <= SAMPLE
    idx = np.arange(a.size) if whole else \
        np.sort(np.random.default_rng(seed).choice(a.size, SAMPLE_EXACT if exact else SAMPLE, replace=False))
    d = {key + '/shape': np.array(a.shape, np.int64), key + '/idx': idx.astype(np.uint32),
         key + '/sample': a.reshape(-1)[idx]}
    if exact and not whole:
        d[key + '/sha256'] = np.array(sha256(a))
    if not exact and not whole:
        s, m = block_sums(a)
        d[key + '/blocksum'], d[key + '/blockabs'] = s, m.astype(np.float32)
    return d


def check(g, key, got, compare):
    """`compare(got_values, stored_values)` on the stored sample, then, for an
    output stored as exact, the digest of all of `got`."""
    got = np.asarray(got)
    assert got.shape == tuple(g[key + '/shape']), (key, got.shape, tuple(g[key + '/shape']))
    compare(got.reshape(-1)[g[key + '/idx']], g[key + '/sample'])
    if key + '/sha256' in g:
        assert sha256(got) == str(g[key + '/sha256']), f'{key}: sample agrees, full output differs'


def check_close(g, key, got, rtol, atol=0.):
    """|got - stored| <= atol + rtol |stored| on the stored sample, and the same
    bound summed over each block on the stored block sums."""
    check(g, key, got, lambda a, b: np.testing.assert_allclose(a, b, rtol=rtol, atol=atol, err_msg=key))
    if key + '/blocksum' in g:
        s, _ = block_sums(got)
        m = g[key + '/blockabs'].astype(np.float64)
        # slack for the float32 rounding of the stored magnitudes and the float64 sums
        bad = np.abs(s - g[key + '/blocksum']) > BLOCK * atol + (rtol * (1 + 1e-6) + 1e-12) * m
        assert not bad.any(), (f'{key}: {int(bad.sum())} of {bad.size} blocks of {BLOCK} values differ by more '
                               f'than the tolerance allows; the first starts at value {int(np.argmax(bad)) * BLOCK}')
