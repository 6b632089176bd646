"""Numpy restatement of the bootstrap draw (csrc/bootstrap.cu) for the tests: Philox4x32-10
(Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC 2011; the round function of
curand_philox4x32_x.h) in vectorised uint64 arithmetic, and a replicate's fragment counts."""
import numpy as np

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
_LO = np.uint64(0xFFFFFFFF)
_32 = np.uint64(32)


def philox4x32_10(ctr, key):
    """ctr: four uint32 words (scalars or arrays), key: two; returns the four output words as
    uint64 arrays.  Products of two 32-bit words fit uint64 exactly."""
    c = [np.asarray(x, dtype=np.uint64) & _LO for x in ctr]
    k0, k1 = [np.asarray(x, dtype=np.uint64) & _LO for x in key]
    for r in range(10):
        p0, p1 = _M0 * c[0], _M1 * c[2]
        c = [(p1 >> _32) ^ c[1] ^ k0, p1 & _LO, (p0 >> _32) ^ c[3] ^ k1, p0 & _LO]
        k0, k1 = (k0 + _W0) & _LO, (k1 + _W1) & _LO
    return c


def mulhi64(r, w):
    """High 64 bits of r * w for uint64 r and w < 2^32, from 32-bit halves (no overflow)."""
    w = np.uint64(w)
    return ((r >> _32) * w + (((r & _LO) * w) >> _32)) >> _32


def boot_counts(w, seed, b):
    """Fragment counts per row of replicate b (int64): W = sum(w) draws, fragment f from
    Philox4x32-10 with counter {f_lo, f_hi, b, 0} and key {seed_lo, seed_hi}; the row is the
    first i whose inclusive prefix sum of w exceeds mulhi64(x0 | x1 << 32, W)."""
    w = np.asarray(w, dtype=np.int64)
    total = int(w.sum())
    f = np.arange(total, dtype=np.uint64)
    seed = np.uint64(seed)
    x = philox4x32_10((f & _LO, f >> _32, np.uint64(b), np.uint64(0)), (seed & _LO, seed >> _32))
    t = mulhi64(x[0] | (x[1] << _32), total)
    rows = np.searchsorted(np.cumsum(w), t.astype(np.int64), side="right")
    return np.bincount(rows, minlength=len(w)).astype(np.int64)
