"""CPU checks of the model behind Corex.sample, impute(return_std=True) and sample_missing: the numpy Philox4x32-10 against
Random123's known answers, and, on the stored goldens for |M| from 0 to n, both paths' conditional standard deviations and
draw maps (tests/dense_sampling.py) against the dense conditional covariance."""
import numpy as np
import pytest

from dense_sampling import dense_conditional_cov, draw_map, lowrank_std
from philox_ref import normals, philox4x32_10, sincospi
from test_conditional_model import NAMES, _masks, _setup


@pytest.mark.parametrize("ctr,key,want", [
    ([0, 0, 0, 0], [0, 0], "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),
    ([0xffffffff] * 4, [0xffffffff] * 2, "408f276d 41c83b0e a20bc7c6 6d5451fd"),
    ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0], "d16cfe09 94fdcceb 5001e420 24126ea1"),
])
def test_philox_known_answers(ctr, key, want):
    got = philox4x32_10(np.array(ctr, dtype=np.uint64), key)
    assert " ".join("%08x" % int(v) for v in got) == want


def test_sincospi_quarter_turns_and_normals():
    x = np.array([0.0, 0.5, 1.0, 1.5, 2.0, 0.25, 1.75])
    s, c = sincospi(x)
    assert np.array_equal(s[:5], [0.0, 1.0, 0.0, -1.0, 0.0]) and np.array_equal(np.abs(c[:5]), [1.0, 0.0, 1.0, 0.0, 1.0])
    assert np.allclose(s, np.sin(np.pi * x), atol=1e-15) and np.allclose(c, np.cos(np.pi * x), atol=1e-15)
    z = normals(7, 0, np.arange(2000), 0, 101)
    assert z.shape == (2000, 101) and abs(z.mean()) < 6 / np.sqrt(z.size) and abs(z.var() - 1) < 6 * np.sqrt(2 / z.size)
    # a stream is its own: another row, draw, tag or seed gives other normals, and fewer columns are a prefix
    assert np.array_equal(normals(7, 0, [5], 0, 40), z[5:6, :40])
    for other in (normals(7, 0, [6], 0, 101), normals(7, 0, [5], 1, 101), normals(7, 1, [5], 0, 101), normals(8, 0, [5], 0, 101)):
        assert not np.any(other == z[5])


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


@pytest.mark.parametrize("name", NAMES)
def test_std_and_draw_maps_match_dense_conditional(name):
    z, x, mean, sd, w = _setup(name)
    m, n = w["B"].shape
    cov = z["covariance"]
    for label, mk in _masks(n, m, 3):
        if not mk.any():
            continue
        want = dense_conditional_cov(cov, sd, mk)
        for path in ("A", "B"):
            std = lowrank_std(w, mk, path)
            assert _rel(std, np.sqrt(np.diag(want))) < 1e-11, (name, label, path, _rel(std, np.sqrt(np.diag(want))))
            mm = draw_map(w, mk, path)
            assert mm.shape == (mk.sum(), mk.sum() + (m if path == "B" else 0))
            assert _rel(mm.dot(mm.T), want) < 1e-11, (name, label, path, _rel(mm.dot(mm.T), want))
        if mk.all():  # nothing observed: the marginal variances, 1 in standardised units
            assert np.abs(lowrank_std(w, mk, "B") ** 2 - 1).max() < 1e-11
