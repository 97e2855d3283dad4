"""CPU checks of the fp8 search's reference (tests/fp8_oracle.py): the properties the quantizer's contract
states, so that the GPU tests compare against a reference that has them."""

from __future__ import annotations

import numpy as np
import torch

import fp8_oracle as F
from oracle import oracle as O


def test_row_scale_lands_in_range():
    rng = np.random.default_rng(0)
    # maxima across bf16's range, and the boundaries of the interval: 224, 448 and their neighbours
    m = O.bf16_round(np.concatenate([10.0 ** rng.uniform(-38, 38, 2000), [1.0, 1.75, 1.7578125, 224.0, 448.0, 449.0, 2.0**-133]]).astype(np.float32))
    m = m[m > 0]
    e = F.row_exponent(m)
    v = m.astype(np.float64) * np.exp2(e.astype(np.float64))
    assert np.all(v > 224) and np.all(v <= 448)
    assert F.row_exponent(np.array([448.0]))[0] == 0 and F.row_exponent(np.array([449.0]))[0] == -1
    assert F.row_exponent(np.array([0.0]))[0] == 0


def test_quantize_max_is_in_range_and_padding_is_zero():
    rng = np.random.default_rng(1)
    for d in (8, 37, 72, 1280):
        x = O.bf16_round((rng.standard_normal((50, d)) * 10.0 ** rng.uniform(-20, 20, (50, 1))).astype(np.float32))
        q, rn = F.quantize(x)
        assert q.shape == (50, F.fp8_width(d)) and q.shape[1] % 16 == 0
        assert np.all(q[:, d:] == 0)
        v = F.dequantize(q)
        assert np.all(np.abs(v).max(axis=1) >= 224) and np.all(np.abs(v).max(axis=1) <= 448)
        assert np.allclose(rn, 1.0 / np.linalg.norm(v.astype(np.float64), axis=1), rtol=1e-6)
        # the quantized cosine is close to the bf16 one (rms error ~1.4e-3 per score at d = 1280)
        cos_q = (v[:, :d] @ v[0, :d]) * rn * rn[0]
        xn = x / np.linalg.norm(x.astype(np.float64), axis=1, keepdims=True)
        assert np.abs(cos_q - xn @ xn[0]).max() < 0.05


def test_zero_rows_stay_zero():
    x = np.zeros((3, 40), np.float32)
    x[1, 5] = -0.0
    q, rn = F.quantize(x)
    assert np.all(F.dequantize(q) == 0)
    assert np.all(rn == np.float32(1e12))


def test_tiny_elements_become_subnormal_or_zero():
    x = np.zeros((1, 32), np.float32)
    x[0, 0] = 1.0  # scaled to 256
    x[0, 1] = 2.0**-12  # 2^-4: normal
    x[0, 2] = 2.0**-15  # 2^-7: subnormal (E4M3's normals end at 2^-6)
    x[0, 3] = 3 * 2.0**-17  # 3 * 2^-9: the subnormal 0x03
    x[0, 4] = 2.0**-18  # 2^-10: half the smallest subnormal, ties to even -> 0
    x[0, 5] = 1.5 * 2.0**-18  # rounds up to the smallest subnormal
    q, _ = F.quantize(O.bf16_round(x))
    assert q[0, 0] == 0x78  # 256 = 1.0 * 2^8
    assert q[0, 1] == 0x18  # 2^-4 = exponent field 3
    assert q[0, 2] == 0x04 and q[0, 3] == 0x03 and q[0, 4] == 0x00 and q[0, 5] == 0x01


def test_power_of_two_multiples_quantize_to_identical_bytes():
    rng = np.random.default_rng(2)
    x = O.bf16_round(rng.standard_normal((20, 100)).astype(np.float32))
    scales = np.exp2(rng.integers(-30, 30, (20, 1))).astype(np.float32)
    a, ra = F.quantize(x)
    b, rb = F.quantize(x * scales)
    assert np.array_equal(a, b) and np.array_equal(ra, rb)


def test_matches_torch_cast_and_round_to_nearest_even():
    # 0x58 = 1.0 * 2^4 = 16 and 0x59 = 18: 17 is the tie and goes to the even mantissa (16)
    v = torch.tensor([17.0, 19.0, 448.0, 240.0]).to(torch.float8_e4m3fn).view(torch.uint8).tolist()
    assert v == [0x58, 0x5A, 0x7E, 0x77]


def test_rescore_reference_skips_padding_and_duplicates():
    rng = np.random.default_rng(3)
    store = O.bf16_round(rng.standard_normal((30, 16)).astype(np.float32))
    q = O.bf16_round(rng.standard_normal((2, 16)).astype(np.float32))
    cand = np.array([[5, -1, 5, 7, 200], [-1, -1, -1, -1, -1]])
    s, i = F.rescore(store, q, cand, 4)
    assert sorted(i[0, :2].tolist()) == [5, 7] and i[0, 2:].tolist() == [-1, -1]
    assert np.all(np.isneginf(s[1])) and np.all(i[1] == -1)
