"""TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  Numpy restatement of the counter-based inter-layer dropout
generator of the flagship training kernels: ``fmix32`` and ``dropout_keep8`` (csrc/na_tc_common.cuh) and the byte layout
``dropout_mask_kernel`` (csrc/na_train_tc.cu) writes.

Window-row ``grow = t * Bp + b`` and unit block ``blk`` (units ``blk * 8 .. blk * 8 + 7`` of the 48) hash to one 32-bit
base word; four more hashes of it give eight 16-bit draws, and unit ``blk * 8 + u`` is kept when its draw is below
``thresh16`` (P(keep) = thresh16 / 65536).  The low and high 32 bits of the 64-bit seed enter the hash separately.

All arithmetic is on uint64 arrays reduced modulo 2**32 after every step, so nothing depends on numpy's overflow rules.
"""
import numpy as np

_M32 = np.uint64(0xFFFFFFFF)
_GOLDEN_B1 = np.uint64(0x9E3779B1)
_GOLDEN_B9 = np.uint64(0x9E3779B9)


def fmix32(h: np.ndarray) -> np.ndarray:
    """MurmurHash3's 32-bit finaliser on uint64 arrays holding 32-bit values."""
    h = np.asarray(h, dtype=np.uint64) & _M32
    h = h ^ (h >> np.uint64(16))
    h = (h * np.uint64(0x85EBCA6B)) & _M32
    h = h ^ (h >> np.uint64(13))
    h = (h * np.uint64(0xC2B2AE35)) & _M32
    return h ^ (h >> np.uint64(16))


def dropout_keep8(seed: int, grow: np.ndarray, blk: np.ndarray, thresh16: int) -> np.ndarray:
    """Keep-bits (bit u = unit blk * 8 + u) of window-row ``grow`` and block ``blk`` (broadcast together) -> uint64 array."""
    if not 0 <= seed < 2 ** 64:
        raise ValueError("seed must be a uint64")
    if not 0 <= thresh16 <= 65536:
        raise ValueError("thresh16 must be in [0, 65536]")
    s = np.uint64(seed)
    idx = np.asarray(grow, dtype=np.uint64) * np.uint64(6) + np.asarray(blk, dtype=np.uint64)   # < 2**64: no wrap needed
    lo = ((idx & _M32) ^ (s & _M32)) * _GOLDEN_B1 & _M32
    hi = (idx >> np.uint64(32)) ^ (s >> np.uint64(32))
    base = fmix32((lo + hi) & _M32)
    th = np.uint64(thresh16)
    bits = np.zeros(base.shape, dtype=np.uint64)
    for i in range(4):
        w = fmix32((base + np.uint64(i + 1) * _GOLDEN_B9) & _M32)
        bits |= ((w & np.uint64(0xFFFF)) < th).astype(np.uint64) << np.uint64(2 * i)
        bits |= ((w >> np.uint64(16)) < th).astype(np.uint64) << np.uint64(2 * i + 1)
    return bits


def dropout_mask_u8(seed: int, thresh16: int, T: int, Bp: int) -> np.ndarray:
    """The keep-mask of (seed, thresh16) as ``na_dropout_mask_u8`` writes it: u8 [T][Bp][48], 1 = kept."""
    grow = np.arange(T * Bp, dtype=np.uint64)[:, None]
    keep = dropout_keep8(seed, grow, np.arange(6, dtype=np.uint64)[None, :], thresh16)      # [T*Bp, 6]
    units = (keep[:, :, None] >> np.arange(8, dtype=np.uint64)) & np.uint64(1)               # [T*Bp, 6, 8]
    return units.astype(np.uint8).reshape(T, Bp, 48)
