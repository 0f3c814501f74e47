"""The dense GEMM's operand split into three bf16 planes, restated in numpy.

x0 = RN_satfinite(x), r = (x - x0) * 2^8, x1 = RN_satfinite(r), x2 = RN_satfinite((r - x1) * 2^8):
the transform of the emulated FastF32 mainloop, which the plane producers (rtf_split_bf16x3)
restate bit for bit.  The GPU tests compare the device split with split_ref."""
import numpy as np

BF16_MAX = np.uint32(0x7F7F0000).view(np.float32)
S = 8


def rn_bf16_satfinite(x: np.ndarray) -> np.ndarray:
    """fp32 -> bf16 (returned as the bf16's fp32 value): round to nearest even, magnitudes past
    the largest finite bf16 (infinities included) clamp to it.  NaN is not handled."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    r = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    out = r.astype(np.uint32).view(np.float32).copy()
    big = ~np.isfinite(out)
    out[big] = np.copysign(BF16_MAX, x[big])
    return out


def split_ref(x: np.ndarray):
    """x (fp32) -> (x0, x1, x2) as fp32 arrays holding bf16 values."""
    x = np.asarray(x, dtype=np.float32)
    s = np.float32(1 << S)
    with np.errstate(over="ignore", invalid="ignore"):
        x0 = rn_bf16_satfinite(x)
        r = (x - x0) * s
        x1 = rn_bf16_satfinite(r)
        x2 = rn_bf16_satfinite((r - x1) * s)
    return x0, x1, x2


def bf16_bits(v: np.ndarray) -> np.ndarray:
    """bit patterns of fp32 arrays holding bf16 values"""
    return (np.asarray(v, dtype=np.float32).view(np.uint32) >> 16).astype(np.uint16)


def edge_values(rng, n=1 << 16) -> np.ndarray:
    """signs, zeros, denormals, bf16 rounding ties and magnitudes up to the largest bf16"""
    e = rng.integers(-149, 128, n).astype(np.float64)
    x = (rng.uniform(1.0, 2.0, n) * np.exp2(e)).astype(np.float32)
    x[np.abs(x) > BF16_MAX] = BF16_MAX
    x *= rng.choice(np.array([-1.0, 1.0], np.float32), n)
    special = np.array([0.0, -0.0, 1.0, -1.0, 2.0 ** -149, -(2.0 ** -149), 2.0 ** -126,
                        1.0 + 2.0 ** -8, 1.0 + 3 * 2.0 ** -8, 1.0 - 2.0 ** -24, BF16_MAX, -BF16_MAX,
                        np.float32(np.pi)], np.float32)
    ties = (rng.integers(0, 1 << 15, 256).astype(np.uint32) << 16 | 0x8000).view(np.float32)
    return np.concatenate([special, ties[np.isfinite(ties)], x]).astype(np.float32)


def test_split_reconstructs_to_fp32():
    """x0 + x1 2^-8 + x2 2^-16 recovers x to within 2^-24 |x| (one fp32 ulp), down to denormals"""
    x = edge_values(np.random.default_rng(0))
    x0, x1, x2 = split_ref(x)
    back = x0.astype(np.float64) + x1 * 2.0 ** -S + x2 * 2.0 ** (-2 * S)
    err = np.abs(back - x.astype(np.float64))
    assert np.all(err <= 2.0 ** -24 * np.abs(x) + 2.0 ** -149)


def test_split_planes_are_bf16_and_ordered():
    x = edge_values(np.random.default_rng(1))
    x0, x1, x2 = split_ref(x)
    for p in (x0, x1, x2):
        assert np.all(p.view(np.uint32) & 0xFFFF == 0)           # exactly bf16
        assert np.all(np.isfinite(p))
    nz = np.abs(x0) >= 2.0 ** -126
    # each further plane carries what the one before could not: at most half a bf16 ulp, scaled
    # (for normal x0; below 2^-126 the ulp is absolute)
    assert np.all(np.abs(x1[nz]) <= np.abs(x0[nz]) * 2.0 ** (S - 8))
    assert np.array_equal(x0[x == 0], x[x == 0]) and np.all(x1[x == 0] == 0)


def test_rounding_is_nearest_even_and_saturating():
    one = np.float32(1.0)
    ulp = np.float32(2.0 ** -7)
    x = np.array([one + ulp / 2, one + 3 * ulp / 2, np.inf, -np.inf, 3.4e38], np.float32)
    got = rn_bf16_satfinite(x)
    assert got[0] == one and got[1] == one + 2 * ulp
    assert got[2] == BF16_MAX and got[3] == -BF16_MAX and got[4] == BF16_MAX
