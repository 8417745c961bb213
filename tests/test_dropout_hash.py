"""The numpy restatement of the in-kernel dropout generator (oracle/dropout_hash.py) on its own: a scalar restatement in
plain Python ints, the two ends of thresh16, the keep rate per unit and per time step, and the seed's high word.
tests/test_gpu_dropout.py pins the CUDA generator to it bit for bit."""
import numpy as np
import pytest

from oracle import dropout_hash as dh

SEEDS = [0, 1, 2 ** 32 - 1, 2 ** 32, 0x2F6B_91C3_5A07_D4E9, 2 ** 64 - 1]


def _fmix32(h):
    h ^= h >> 16
    h = (h * 0x85EBCA6B) & 0xFFFFFFFF
    h ^= h >> 13
    h = (h * 0xC2B2AE35) & 0xFFFFFFFF
    return h ^ (h >> 16)


def _keep8(seed, grow, blk, thresh16):
    """dropout_keep8 of csrc/na_tc_common.cuh, one block at a time on Python ints."""
    idx = (grow * 6 + blk) & 0xFFFFFFFFFFFFFFFF
    base = _fmix32(((((idx ^ seed) & 0xFFFFFFFF) * 0x9E3779B1) + ((idx >> 32) ^ (seed >> 32))) & 0xFFFFFFFF)
    bits = 0
    for i in range(4):
        w = _fmix32((base + (i + 1) * 0x9E3779B9) & 0xFFFFFFFF)
        bits |= int((w & 0xFFFF) < thresh16) << (2 * i)
        bits |= int((w >> 16) < thresh16) << (2 * i + 1)
    return bits


@pytest.mark.parametrize("seed", SEEDS)
def test_vectorised_equals_scalar_restatement(seed):
    T, Bp, th = 3, 37, 26214
    mask = dh.dropout_mask_u8(seed, th, T, Bp)
    assert mask.shape == (T, Bp, 48) and mask.dtype == np.uint8
    for t in range(T):
        for b in range(Bp):
            for blk in range(6):
                bits = _keep8(seed, t * Bp + b, blk, th)
                assert [int(v) for v in mask[t, b, blk * 8:blk * 8 + 8]] == [(bits >> u) & 1 for u in range(8)], (t, b, blk)
    # rows past 2**32 / 6: the high word of the row index enters the hash
    grow = np.array([2 ** 32 // 6 - 1, 2 ** 32 // 6 + 1, 3 * 2 ** 40 + 7], dtype=np.uint64)
    for g in grow:
        for blk in range(6):
            assert int(dh.dropout_keep8(seed, g, blk, th)) == _keep8(seed, int(g), blk, th)


@pytest.mark.parametrize("seed", SEEDS)
def test_thresh16_ends_drop_all_and_keep_all(seed):
    assert not dh.dropout_mask_u8(seed, 0, 5, 130).any()
    assert dh.dropout_mask_u8(seed, 65536, 5, 130).all()
    assert dh.dropout_mask_u8(seed, 1, 5, 130).sum() < 10          # P(keep) = 1 / 65536 per unit


@pytest.mark.parametrize("thresh16", [1311, 26214, 32768, 62259])
def test_keep_rate_per_unit_and_per_step(thresh16):
    """Every unit index (over all rows) and every time step (over all windows and units) keeps at thresh16 / 65536, within
    5 sigma of the binomial spread."""
    T, Bp = 64, 512
    mask = dh.dropout_mask_u8(0x1234_5678_9ABC_DEF0, thresh16, T, Bp).astype(np.float64)
    q = thresh16 / 65536
    per_unit = mask.mean(axis=(0, 1))
    assert np.abs(per_unit - q).max() < 5 * np.sqrt(q * (1 - q) / (T * Bp)), per_unit
    per_step = mask.mean(axis=(1, 2))
    assert np.abs(per_step - q).max() < 5 * np.sqrt(q * (1 - q) / (Bp * 48)), per_step


def test_seed_high_and_low_words_both_change_the_mask():
    T, Bp, th = 4, 256, 26214
    q = th / 65536
    base = dh.dropout_mask_u8(5, th, T, Bp)
    for other in (5 + 2 ** 32, 5 + 2 ** 63, 6, 5 ^ (2 ** 64 - 1)):
        frac = (dh.dropout_mask_u8(other, th, T, Bp) != base).mean()
        assert abs(frac - 2 * q * (1 - q)) < 0.03, (other, frac)      # independent masks differ at rate 2q(1-q)


def test_rejects_out_of_range_arguments():
    with pytest.raises(ValueError):
        dh.dropout_mask_u8(2 ** 64, 100, 1, 1)
    with pytest.raises(ValueError):
        dh.dropout_mask_u8(-1, 100, 1, 1)
    with pytest.raises(ValueError):
        dh.dropout_mask_u8(0, 65537, 1, 1)
