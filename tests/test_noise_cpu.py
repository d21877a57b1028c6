"""CPU: the numpy restatement of the keyed noise stream (oracle/philox.py) -- Philox4x32-10 known answers, the layout and
offset identities the sampler's keyed calls rely on, and the statistics of the normals."""
import numpy as np
import pytest
from scipy import stats

from oracle import philox as P


def _hex(x):
    return [int(v) for v in x]


@pytest.mark.parametrize("ctr,key,want", [
    ([0, 0, 0, 0], [0, 0], [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]),
    ([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2, [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]),
    ([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0],
     [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]),
])
def test_philox_known_answers(ctr, key, want):
    got = P.philox4x32_10(np.array(ctr, dtype=np.uint32), np.array(key, dtype=np.uint32))
    assert _hex(got) == want


def test_normal_known_values():
    z = P.normal(0, 0, 0, 0, np.arange(6))
    np.testing.assert_allclose(z, [0.991138, -0.924663, -0.617609, -0.482068, -0.153638, 0.180826], atol=1e-6)
    z = P.normal(0x0123456789ABCDEF, 3, 1000000, 4, np.array([0, 1, 84]))
    np.testing.assert_allclose(z, [-0.449827, -0.401344, -0.664848], atol=1e-6)


def test_key_words():
    assert _hex(P.seed_key(0x0123456789ABCDEF)) == [0x89ABCDEF, 0x01234567]
    assert _hex(P.seed_key(-1)) == [0xFFFFFFFF, 0xFFFFFFFF]


def test_pose_offset_identity():
    """A piece of a call that starts at pose 3 draws rows 3..6 of the whole call, for every hypothesis."""
    whole = P.noise(11, 3, 10, 2)
    part = P.noise(11, 3, 4, 2, pose_offset=3)
    w = whole.reshape(3, 2, 10, 17, 5)[:, :, 3:7]
    np.testing.assert_array_equal(part.reshape(3, 2, 4, 17, 5), w)


def test_step_offset_identity():
    whole = P.noise(12, 6, 5, 3)
    for k in range(6):
        np.testing.assert_array_equal(P.noise(12, 1, 5, 3, step_offset=k)[0], whole[k])


def test_hypothesis_major_order():
    n, H = 7, 3
    z = P.noise(13, 2, n, H)
    for h in range(H):
        for p in range(n):
            want = P.normal(13, np.arange(2)[:, None], p, h, np.arange(85)[None, :]).reshape(2, 17, 5)
            np.testing.assert_array_equal(z[:, h * n + p], want)


def test_seed_high_word_matters():
    a = P.noise(5, 2, 8, 1)
    b = P.noise(5 + (1 << 32), 2, 8, 1)
    c = P.noise(5 + (7 << 40), 2, 8, 1)
    assert np.mean(a == b) < 1e-3 and np.mean(a == c) < 1e-3 and np.mean(b == c) < 1e-3


def test_counter_covers_every_element_once():
    """Each quad feeds four consecutive elements with distinct words: lanes 0/1 share (x0, x1) through cos / sin, lanes
    2/3 share (x2, x3); no two elements of a row are equal."""
    z = P.noise(14, 1, 64, 2).reshape(-1, 85)
    for row in z:
        assert len(np.unique(row)) == 85


def test_statistics():
    """2^22+ normals over steps, hypotheses, poses and elements: moments, KS against N(0, 1), and lag-1 correlations
    along e, s, b and h."""
    S, H, B = 16, 4, 1024
    z = P.noise(0x5EED, S, B, H)                  # [S, H*B, 17, 5]
    assert z.size >= 1 << 22
    v = z.ravel()
    n = v.size
    assert abs(v.mean()) < 5 / np.sqrt(n)
    assert abs(v.var() - 1.0) < 5 * np.sqrt(2.0 / n)
    assert abs(stats.skew(v)) < 5 * np.sqrt(6.0 / n)
    assert abs(stats.kurtosis(v)) < 5 * np.sqrt(24.0 / n)
    assert stats.kstest(v, "norm").pvalue > 1e-4
    g = z.reshape(S, H, B, 85)

    def lag_corr(a, b):
        a, b = a.ravel(), b.ravel()
        return np.corrcoef(a, b)[0, 1], a.size

    for name, (a, b) in {
        "e": (g[..., :-1], g[..., 1:]),
        "e+2": (g[..., :-2], g[..., 2:]),
        "s": (g[:-1], g[1:]),
        "h": (g[:, :-1], g[:, 1:]),
        "b": (g[:, :, :-1], g[:, :, 1:]),
    }.items():
        r, m = lag_corr(a, b)
        assert abs(r) < 5 / np.sqrt(m), f"lag correlation along {name}: {r:.2e}"
