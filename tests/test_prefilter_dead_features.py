"""CPU checks of the prefilter's dead-feature skip (no GPU needed): the feature permutation the library applies to the
embedded network (dsmppi_permute_hidden) is an exact transform of it, and anything but a permutation is rejected."""
import ctypes as C

import numpy as np
import pytest


@pytest.fixture(scope="module")
def lib():
    from optimalmodulationds_b200 import build, _capi
    build.build()
    return _capi.load()


def _frame(rng, O):
    W = np.concatenate([rng.standard_normal(3 * 256 * 256), rng.standard_normal(O * 256)]).astype(np.float32) * 0.1
    b = rng.standard_normal(3 * 256 + O).astype(np.float32) * 0.1
    return W, b


def _forward(W, b, O, h1):
    """layers 2..5 in fp64 from first-layer activations h1 (rows)"""
    h = h1.astype(np.float64)
    W, b = W.astype(np.float64), b.astype(np.float64)
    for l in range(3):
        h = np.maximum(h @ W[l * 65536:(l + 1) * 65536].reshape(256, 256).T + b[l * 256:(l + 1) * 256], 0.0)
    return h @ W[3 * 65536:].reshape(O, 256).T + b[768:]


def test_permuted_network_equals_the_original(lib):
    rng = np.random.default_rng(3)
    O = 9
    W, b = _frame(rng, O)
    perm = np.concatenate([rng.permutation(256) for _ in range(3)]).astype(np.int32)
    Wp, bp = np.empty_like(W), np.empty_like(b)
    assert lib.dsmppi_permute_hidden(O, W.ctypes.data, b.ctypes.data, perm.ctypes.data, Wp.ctypes.data,
                                     bp.ctypes.data) == 0
    assert not np.array_equal(W, Wp)
    h1 = np.maximum(rng.standard_normal((512, 256)), 0.0)
    ref, out = _forward(W, b, O, h1), _forward(Wp, bp, O, h1)
    # the same products summed in another order: equal to fp64 rounding
    assert np.allclose(out, ref, rtol=1e-12, atol=1e-12 * np.abs(ref).max())


def test_a_non_permutation_is_rejected(lib):
    O = 2
    W, b = _frame(np.random.default_rng(0), O)
    perm = np.tile(np.arange(256, dtype=np.int32), 3)
    perm[300] = perm[301]
    out_W, out_b = np.empty_like(W), np.empty_like(b)
    assert lib.dsmppi_permute_hidden(O, W.ctypes.data, b.ctypes.data, perm.ctypes.data, out_W.ctypes.data,
                                     out_b.ctypes.data) == 2
