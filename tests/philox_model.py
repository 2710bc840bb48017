"""CPU model of the production random numbers -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The production path draws every random number from Philox4x32-10 (`csrc/philox.cuh`), addressed by what it is for
(DESIGN.md §2, deviation 2), keyed by the 64-bit seed ``(seed_lo, seed_hi)``:

* Fano normal of (event, nucleus index, grid step k): counter ``(event_lo, event_hi, nucleus, k)``, Box-Muller in
  single precision;
* time-bucket wiggle of (event, Szudzik key): counter ``(event_lo, event_hi, 0xFFFFFFFF, key)``, 16 bits.

This module restates them from the definition of Salmon et al., "Parallel random numbers: as easy as 1, 2, 3" (SC'11),
for `tests/test_philox_model.py` and `tests/test_gpu_production.py`.
"""

from __future__ import annotations

import numpy as np

PHILOX_M0, PHILOX_M1 = 0xD2511F53, 0xCD9E8D57  # round multipliers
PHILOX_W0, PHILOX_W1 = 0x9E3779B9, 0xBB67AE85  # key schedule (Weyl) increments
STREAM_WIGGLE = 0xFFFFFFFF
NORMAL_ABS_MAX = 8.66  # the draw gate: mean + spread * NORMAL_ABS_MAX >= 1

_U32 = np.uint64(0xFFFFFFFF)
_S32 = np.uint64(32)


def _u32(a):
    return np.asarray(a, dtype=np.uint64) & _U32


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32 with 10 rounds, vectorised over numpy arrays of 32-bit words; returns four uint32 arrays.

    One round: (hi0, lo0) = M0 * c0, (hi1, lo1) = M1 * c2 (64-bit products);
    c <- (hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0); then the key is bumped by the Weyl increments."""
    c0, c1, c2, c3, k0, k1 = np.broadcast_arrays(*(_u32(a) for a in (c0, c1, c2, c3, k0, k1)))
    c0, c1, c2, c3, k0, k1 = (a.copy() for a in (c0, c1, c2, c3, k0, k1))
    m0, m1 = np.uint64(PHILOX_M0), np.uint64(PHILOX_M1)
    w0, w1 = np.uint64(PHILOX_W0), np.uint64(PHILOX_W1)
    for _ in range(10):
        p0 = m0 * c0  # < 2^64: exact in uint64
        p1 = m1 * c2
        c0, c1, c2, c3 = (p1 >> _S32) ^ c1 ^ k0, p1 & _U32, (p0 >> _S32) ^ c3 ^ k1, p0 & _U32
        k0 = (k0 + w0) & _U32
        k1 = (k1 + w1) & _U32
    return tuple(a.astype(np.uint32) for a in (c0, c1, c2, c3))


def _counter(seed, event, stream, index):
    """Philox counter and key of a draw; ``seed`` and ``event`` are 64-bit (Python ints or uint64 arrays)."""
    seed = np.asarray(int(seed) & (2**64 - 1) if isinstance(seed, int) else seed, dtype=np.uint64)
    event = np.asarray(event, dtype=np.uint64)
    return (event & _U32, event >> _S32, stream, index, seed & _U32, seed >> _S32)


def uniform53(a, b):
    """53-bit uniform in [0, 1) from two words, numpy's next_double recipe: ((a >> 5) 2^26 + (b >> 6)) / 2^53."""
    a, b = np.asarray(a, dtype=np.uint64), np.asarray(b, dtype=np.uint64)
    return ((a >> np.uint64(5)) << np.uint64(26) | (b >> np.uint64(6))).astype(np.float64) * 2.0**-53


def philox_uniform(seed, event, stream, index):
    x = philox4x32_10(*_counter(seed, event, stream, index))
    return uniform53(x[0], x[1])


def philox_uniform16(seed, event, stream, index):
    x = philox4x32_10(*_counter(seed, event, stream, index))
    return (x[0] >> np.uint32(16)).astype(np.float64) / 65536.0


def wiggle16(seed, event, key):
    """The time-bucket wiggle of Szudzik key ``key`` in event ``event``: k / 2^16, k the top 16 bits of word 0."""
    return philox_uniform16(seed, event, STREAM_WIGGLE, key)


def box_muller(u53, x2):
    """(z_ref, z_err) of the device's single-precision Box-Muller from its two inputs, see `fano_normal`."""
    u1 = (np.asarray(u53, dtype=np.float64) + 2.0**-54).astype(np.float32).astype(np.float64)  # (0, 1], cast RN
    u2 = (np.asarray(x2, dtype=np.uint32) >> np.uint32(8)).astype(np.float64) / 2.0**24  # exact
    z = np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)
    return z, 1e-6 * np.abs(z) + 1e-9


def fano_normal(seed, event, nucleus, step):
    """The Fano normal of (event, nucleus, grid step) as ``(z_ref, z_err)``: |z_device - z_ref| <= z_err.

    The device (`philox_normal`) computes, from the Philox words x0..x3,
      u1 = (float)(uniform53(x0, x1) + 2^-54)   (the double sum is exact or rounded the same on both sides; the cast
                                                 to float rounds to nearest -- both reproduced here bit for bit)
      u2 = (x2 >> 8) * 2^-24                    (exact in float)
      z  = sqrtf(-2 logf(u1)) * cospif(2 u2)    (float32), widened to double.
    z_ref evaluates the last line in float64 on the same u1, u2.  The library is built without -use_fast_math, so
    `sqrtf` and the products are correctly rounded (relative error <= 2^-24 each) and `logf`, `cospif` are within
    1 ulp (relative <= 2^-23).  -2 logf is exact; the square root halves the relative error of its argument.  In all
      |z - z_ref| / |z_ref| <= 2^-24 (log, halved) + 2^-24 (sqrt) + 2^-23 (cospi) + 2^-24 (product) = 5 * 2^-24 ~ 3e-7
    to first order, plus the float64 rounding of z_ref itself (~1e-16 |z| relative, and ~1e-15 absolute where
    cos(2 pi u2) passes through zero).  ``z_err = 1e-6 |z_ref| + 1e-9`` covers that with a factor of three to spare.
    """
    x = philox4x32_10(*_counter(seed, event, nucleus, step))
    return box_muller(uniform53(x[0], x[1]), x[2])
