"""CPU checks of tests/slice_reference.py, the node-by-node statement of the elliptical-slice update that the GPU tests of
nhp_cont_resample_baseline compare against: driven by the same z and u, it must give the curves of the host mirror
LogGaussianCoxProcess.resample_ (run with a scripted generator and a NumPy likelihood).  This pins the random-number layout of the
C ABI (z[g + G k], u[j + 101 k]) to the host algorithm."""
import types

import numpy as np
import pytest

import slice_reference as sr
from nhp_b200.continuous import LogGaussianCoxProcess


def _problem(K, G, T, seed, n_events, empty=()):
    rng = np.random.default_rng(seed)
    x = np.linspace(0.0, T, G)
    lam = np.exp(0.3 * np.sin(rng.uniform(0.5, 3.0, (K, 1)) * x[None, :] / T * 6.0 + rng.uniform(0, 6, (K, 1))))
    tb = [np.sort(rng.uniform(0.0, T, rng.integers(0, n_events))) for _ in range(K)]
    for k in empty:
        tb[k] = np.zeros(0)
    z = rng.standard_normal((K, G))
    u = rng.random((K, sr.NU))
    return x, lam, tb, z, u


def _mirror(x, lam, tb, z, u, m=0.0, eta=None):
    b = LogGaussianCoxProcess(x, lam.copy(), m=m, sigma=1.0, eta=eta or (x[-1] - x[0]) / 10.0)
    ctx = sr.NumpyLoglikContext(x, tb)
    out = b.resample_(ctx, types.SimpleNamespace(h=None), sr.ScriptedRng(z, u))
    return b, out, ctx.calls


@pytest.mark.parametrize("K,G,m,empty", [(3, 2, 0.0, ()), (6, 37, 0.2, (2,)), (4, 600, -0.1, ())])
def test_statement_equals_the_mirror(K, G, m, empty):
    x, lam, tb, z, u = _problem(K, G, 50.0, 7 + G, 60, empty)
    b, out, calls = _mirror(x, lam, tb, z, u, m=m)
    ref, att = sr.slice_update(x, lam, b._chol, m, tb, z, u)
    np.testing.assert_allclose(out, ref, rtol=1e-13)
    # the mirror evaluates every node once per round: round 0 plus as many rounds as the slowest node's attempts
    assert calls == 1 + att.max()
    assert np.all(att >= 1)


def test_rejections_shrink_the_bracket_the_same_way():
    """Slice heights near 1 and little data: several attempts per node, each drawing from the shrunken bracket."""
    K, G = 8, 11
    x, lam, tb, z, u = _problem(K, G, 40.0, 3, 400)
    u[:, 0] = 1.0 - 1e-9
    b, out, _ = _mirror(x, lam, tb, z, u)
    ref, att = sr.slice_update(x, lam, b._chol, 0.0, tb, z, u)
    np.testing.assert_allclose(out, ref, rtol=1e-13)
    assert att.max() >= 3


def test_attempt_limit_is_reached_by_both():
    """Angle uniforms of 0 keep theta at the rejected end of the bracket: the first candidate, exp(L z) with large z, is tried again
    and again."""
    K, G = 2, 5
    x, lam, tb, z, u = _problem(K, G, 20.0, 5, 30)
    u[:, 1] = 0.25
    u[:, 2:] = 0.0
    z[:] = 30.0
    L = LogGaussianCoxProcess(x, lam, eta=2.0)._chol
    with pytest.raises(RuntimeError, match="maximum attempts"):
        sr.slice_update(x, lam, L, 0.0, tb, z, u)
    with pytest.raises(RuntimeError, match="maximum attempts"):
        _mirror(x, lam, tb, z, u)
