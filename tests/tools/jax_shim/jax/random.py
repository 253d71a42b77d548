"""jax.random for jax==0.4.8 (threefry2x32, jax_threefry_partitionable=False) in pure NumPy.

Written from the published algorithm (jax/_src/prng.py, jax/_src/random.py at v0.4.8),
independently of oracle/rbg_oracle.c; both are checked against the same reference-owned
golden vectors (tests/golden/reference_goldens.json).
"""
import math

import numpy as _np

from ._core import asarr

_U32 = _np.uint32
_ROT = ((13, 15, 26, 6), (17, 29, 16, 24))


def _rotl(x, r):
    return (x << _U32(r)) | (x >> _U32(32 - r))


def threefry2x32(k0, k1, x0, x1):
    """Random123 Threefry-2x32, 20 rounds, element-wise over the counter arrays."""
    with _np.errstate(over="ignore"):
        k0, k1 = _U32(k0), _U32(k1)
        x0 = _np.array(x0, dtype=_U32, copy=True).reshape(-1)
        x1 = _np.array(x1, dtype=_U32, copy=True).reshape(-1)
        ks = (k0, k1, _U32(k0 ^ k1 ^ _U32(0x1BD11BDA)))
        x0 = x0 + ks[0]
        x1 = x1 + ks[1]
        for g in range(5):
            for r in _ROT[g & 1]:
                x0 = x0 + x1
                x1 = _rotl(x1, r)
                x1 = x1 ^ x0
            x0 = x0 + ks[(g + 1) % 3]
            x1 = x1 + ks[(g + 2) % 3] + _U32(g + 1)
    return x0, x1


def _threefry_iota(key, n):
    """threefry_2x32(key, iota(n)): odd sizes are padded with one zero, halves are the two counter words."""
    key = _np.asarray(key, dtype=_U32).reshape(2)
    counts = _np.arange(n, dtype=_U32)
    if n % 2:
        counts = _np.concatenate([counts, _np.zeros(1, _U32)])
    h = counts.size // 2
    o0, o1 = threefry2x32(key[0], key[1], counts[:h], counts[h:])
    return _np.concatenate([o0, o1])[:n]


def PRNGKey(seed):
    seed = int(seed)
    return asarr(_np.array([(seed >> 32) & 0xFFFFFFFF, seed & 0xFFFFFFFF], dtype=_U32))


def split(key, num=2):
    return asarr(_threefry_iota(key, 2 * int(num)).reshape(int(num), 2))


def _shape(shape):
    if isinstance(shape, (tuple, list)):
        return tuple(int(s) for s in shape)
    return (int(shape),)


def _random_bits(key, shape):
    shape = _shape(shape)
    n = int(_np.prod(shape)) if shape else 1
    return _threefry_iota(key, n).reshape(shape)


def uniform(key, shape=(), dtype=_np.float32, minval=0.0, maxval=1.0):
    bits = _random_bits(key, shape)
    f = ((bits >> _U32(9)) | _U32(0x3F800000)).view(_np.float32) - _np.float32(1.0)
    lo, hi = _np.float32(minval), _np.float32(maxval)
    f = f * (hi - lo) + lo
    return asarr(_np.maximum(lo, f).reshape(_shape(shape)), _np.float32)


GUMBEL_TRACE = []  # (23-bit mantissas, candidate mask, pick) of every choice(p, replace=False): see make_seqrw_fixtures.py


def gumbel(key, shape=(), dtype=_np.float32):
    """-log(-log(uniform(key, shape, minval=tiny, maxval=1))) in float32 (jax/_src/random.py v0.4.8 `_gumbel`)."""
    u = _np.asarray(uniform(key, shape, minval=_np.finfo(_np.float32).tiny, maxval=1.0))
    with _np.errstate(divide="ignore"):
        return asarr((-_np.log(-_np.log(u))).astype(_np.float32), _np.float32)


def randint(key, shape, minval, maxval, dtype=_np.int32):
    shape = _shape(shape)
    k1, k2 = _np.asarray(split(key))
    hi_bits = _random_bits(k1, shape).astype(_np.uint64)
    lo_bits = _random_bits(k2, shape).astype(_np.uint64)
    minval, maxval = int(minval), int(maxval)
    span = (maxval - minval) & 0xFFFFFFFF
    if maxval <= minval:
        span = 1
    mult = ((65536 % span) ** 2 & 0xFFFFFFFF) % span  # squared in uint32: 2**32 wraps to 0 for span > 2**16
    off = ((hi_bits % span) * mult + (lo_bits % span)) & 0xFFFFFFFF  # uint32 arithmetic wraps
    off = off % span
    return asarr((minval + off.astype(_np.int64)).astype(_np.int32).reshape(shape))


def _shuffle(key, x, axis=0):
    x = _np.asarray(x)
    n = x.shape[axis]
    if n <= 1:
        return asarr(x)
    rounds = int(math.ceil(3 * math.log(max(1, x.size)) / math.log(2**32 - 1)))
    assert axis == 0
    for _ in range(rounds):
        key, sub = _np.asarray(split(key))
        sort_keys = _random_bits(sub, x.shape)
        if x.ndim == 1:
            x = x[_np.argsort(sort_keys, kind="stable")]
        else:  # independent sort along axis 0 of every column
            order = _np.argsort(sort_keys, axis=0, kind="stable")
            x = _np.take_along_axis(x, order, axis=0)
    return asarr(x)


def permutation(key, x, axis=0, independent=False):
    if _np.ndim(x) == 0:
        return _shuffle(key, _np.arange(int(x), dtype=_np.int32), 0)
    x = _np.asarray(x)
    if independent or x.ndim == 1:
        return _shuffle(key, x, axis)
    ind = _np.asarray(_shuffle(key, _np.arange(x.shape[axis], dtype=_np.int32), 0))
    return asarr(_np.take(x, ind, axis=axis))


def choice(key, a, shape=(), replace=True, p=None, axis=0):
    shape = _shape(shape) if not isinstance(shape, tuple) or shape != () else ()
    if _np.ndim(a) == 0:
        a = _np.arange(int(a), dtype=_np.int32)
    a = _np.asarray(a)
    n_inputs = a.shape[axis]
    n_draws = int(_np.prod(shape)) if shape else 1
    if n_draws == 0:
        return asarr(_np.zeros(shape, a.dtype))
    if not replace and n_draws > n_inputs:
        raise ValueError("Cannot take a larger sample than population when 'replace=False'")
    if p is None:
        if replace:
            ind = _np.asarray(randint(key, shape, 0, n_inputs))
            result = _np.take(a, ind, axis=axis)
        else:
            perm = _np.asarray(permutation(key, a, axis))
            sl = (slice(None),) * axis + (slice(n_draws),)
            result = perm[sl]
    else:
        p_arr = _np.asarray(p).astype(_np.float32)
        assert p_arr.shape == (n_inputs,)
        if replace:
            p_cuml = _np.cumsum(p_arr, dtype=_np.float32)
            r = p_cuml[-1] * (_np.float32(1.0) - _np.asarray(uniform(key, shape)))
            ind = _np.searchsorted(p_cuml, r.astype(_np.float32), side="left")
            ind = _np.clip(ind, 0, n_inputs - 1)
        else:
            # Gumbel top-k (jax/_src/random.py v0.4.8): g = -gumbel(key, (n,)) - log(p); ind = argsort(g)[:n_draws].
            # SequentialRandomWalkBoard (sequential_random_walk.py:57-63, 211-217) draws every cell this way.
            with _np.errstate(divide="ignore"):
                g = -_np.asarray(gumbel(key, (n_inputs,))) - _np.log(p_arr)
            ind = _np.argsort(g, kind="stable")[:n_draws]
            GUMBEL_TRACE.append((_np.asarray(_random_bits(key, (n_inputs,))) >> _U32(9), p_arr > 0, int(ind[0])))
        result = _np.take(a, ind, axis=axis)
    full_shape = shape if a.ndim == 0 else a.shape[:axis] + tuple(shape) + a.shape[axis + 1:]
    return asarr(_np.asarray(result).reshape(full_shape))
