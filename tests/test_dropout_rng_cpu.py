"""The torch int64 restatement of the dropout RNG (tests/dropout_rng.py), which the GPU tests use to rebuild kernel masks at
full size, against the plain uint64 numpy statement and a published splitmix64 value; the two mask layouts against an
element-by-element statement of their index formulas."""
import numpy as np
import pytest
import torch

import dropout_rng as R

SEEDS = [0, 12345, 0x5EEDA4D2, (1 << 47) | 0x1234567, (1 << 48) - 1]


@pytest.mark.parametrize("seed", SEEDS)
@pytest.mark.parametrize("start", [0, 0x1_2345_6789, (1 << 32) - 32768, (1 << 62) + 7])
def test_torch_rng64_matches_numpy_bit_for_bit(seed, start):
    ctr = np.arange(65536, dtype=np.uint64) + np.uint64(start)
    ref = R.rng64_np(seed, ctr)
    got = R.rng64(seed, torch.arange(65536, dtype=torch.int64) + start).numpy().view(np.uint64)
    assert np.array_equal(got, ref)


def test_rng64_is_splitmix64():
    # splitmix64 seeded with 0 returns 0xE220A8397B1DCDAF first: its state after one step is the golden-ratio increment,
    # i.e. counter 1 with seed 0 here
    assert int(R.rng64_np(0, np.array([1], dtype=np.uint64))[0]) == 0xE220A8397B1DCDAF
    assert int(R.rng64(0, torch.tensor([1])).numpy().view(np.uint64)[0]) == 0xE220A8397B1DCDAF


def test_threshold_and_scale_are_the_kernels_float32_values():
    assert R.thr16(0.1) == 6554 and R.thr16(0.25) == 16384 and R.thr16(0.0) == 0
    assert R.keep_scale(0.1) == float(np.float32(65536.0) / np.float32(65536 - 6554))


def _lane_keep(seed, ctr, lane, p):
    bits = R.rng64_np(seed, np.array([ctr], dtype=np.uint64))[0]
    return int((bits >> np.uint64(16 * lane)) & np.uint64(0xFFFF)) >= R.thr16(p)


@pytest.mark.parametrize("offset", [0, (1 << 32) + 12345])
def test_element_layout(offset):
    seed, p, N = (1 << 47) | 99, 0.1, 72
    rows = torch.tensor([0, 1, 5, 333, (1 << 26) + 3])
    got = R.element_keep(seed, offset, p, rows, N)
    assert tuple(got.shape) == (5, N)
    for a, r in enumerate(rows.tolist()):
        for c in range(N):
            e = r * N + c
            assert bool(got[a, c]) == _lane_keep(seed, offset + e // 4, e % 4, p), (r, c)
    frac = float(R.element_keep(seed, offset, p, torch.arange(4096), 768).float().mean())
    assert abs(frac - 0.9) < 5e-3, frac


@pytest.mark.parametrize("offset", [1000, (1 << 32) + 12345])
def test_attention_probability_layout(offset):
    seed, p, heads, L = (1 << 47) | 4242, 0.1, 3, 30
    seqs = torch.tensor([0, 2, 21503])
    got = R.prob_keep(seed, offset, p, seqs, heads, L)
    assert tuple(got.shape) == (3, heads, L, L)
    for a, n in enumerate(seqs.tolist()):
        for h in range(heads):
            for i in range(L):
                for j in range(L):
                    nt, t, e = j // 8, (j % 8) // 2, j % 2
                    ctr = offset + ((n * heads + h) * 32 + i) * 8 + (nt >> 1) * 4 + t
                    assert bool(got[a, h, i, j]) == _lane_keep(seed, ctr, (nt & 1) * 2 + e, p), (n, h, i, j)
