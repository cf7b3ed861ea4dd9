"""CPU: pin the oracle (oracle/nnk_oracle.c) against the golden vectors generated from the
UNMODIFIED reference (tests/golden/make_golden.py) and against the reference's own known-answer
tests."""
import os

import numpy as np
import pytest

import oracle
from conftest import ROOT, rel_err, windows_set


@pytest.fixture(scope="module")
def parity_golden():
    return np.load(os.path.join(ROOT, "tests", "golden", "reference_parity_golden.npz"))


def test_mlpg_oracle_matches_reference_golden(golden):
    for wi, ws in enumerate(windows_set()):
        for dt in ("float32", "float64"):
            for T in (1, 2, 5, 12):
                key = "w%d_%s_T%d" % (wi, dt, T)
                m, v, go = golden[key + "_means"], golden[key + "_vars"], golden[key + "_go"]
                y = oracle.mlpg(m, v, ws)
                assert y.dtype == m.dtype  # tests/test_paramgen.py:58
                # same arithmetic in the same order -> bit-identical
                assert np.array_equal(y, golden[key + "_y"]), key
                assert np.array_equal(oracle.mlpg(m, v[0].copy(), ws), golden[key + "_y1d"]), key
                g = oracle.mlpg_grad(m, v, ws, go)
                assert g.dtype == np.float32 and g.shape == m.shape
                assert rel_err(g, golden[key + "_grad"]) < 2e-6, key


def test_cfg1_oracle_matches_reference_golden(golden):
    r1 = np.random.default_rng(1234)
    m = r1.random((100, 177)).astype(np.float32)
    v = (r1.random((100, 177)) + 0.1).astype(np.float32)
    ws = windows_set()[2]
    assert np.array_equal(oracle.mlpg(m, v, ws), golden["cfg1_y"])
    assert np.array_equal(oracle.mlpg(m, np.ones(177, dtype=np.float32), ws), golden["cfg1_y_unitvar"])


def test_unit_variance_matrix_oracle(golden):
    for wi, ws in enumerate(windows_set()):
        for T in (3, 10):
            R = oracle.unit_variance_mlpg_matrix(ws, T)
            assert R.dtype == np.float32 and R.shape == (T, len(ws) * T)
            assert np.abs(R - golden["w%d_R_T%d" % (wi, T)]).max() < 1e-7
    assert np.abs(oracle.unit_variance_mlpg_matrix(windows_set()[2], 40) - golden["w2_R_T40"]).max() < 1e-7
    # NB the T=3 matrix printed in the reference's docstring (paramgen/_mlpg.py:335-344) is stale: the
    # reference itself no longer reproduces it (it predates the edge-precision rule of :352-367), so
    # the pin is the reference's actual output stored in the golden file (w2_R_T3 above).


def test_bandmat_known_answers(golden):
    # reference tests/bandmat/test_linalg.py:100-114 (4x4 SPD tridiagonal, lower band storage)
    c = oracle.cholesky_banded_lower(golden["chol4_ab"])
    assert np.array_equal(c, golden["chol4_c"])
    a = np.array([[4.0, 1.0, 0.0, 0.0], [1.0, 4.0, 0.5, 0.0], [0.0, 0.5, 4.0, 0.2], [0.0, 0.0, 0.2, 4.0]])
    lfac = np.zeros_like(a)
    lfac[range(4), range(4)] = c[0]
    lfac[(1, 2, 3), (0, 1, 2)] = c[1, :3]
    assert np.allclose(a, lfac @ lfac.T, rtol=1e-7, atol=1e-14)
    x = oracle.cho_solve_lower(c, np.array([1.0, 2.0, 3.0, 4.0]))
    assert np.allclose(a @ x, [1.0, 2.0, 3.0, 4.0])
    # non positive definite -> LinAlgError naming the 1-based frame (linalg.pyx:79-82)
    with pytest.raises(np.linalg.LinAlgError, match="2-th leading minor"):
        oracle.cholesky_banded_lower(np.array([[1.0, 0.5, 1.0], [1.0, 0.0, 0.0]]))
    # cholesky_inv_banded, reference tests/test_util.py:62-81
    assert np.allclose(oracle.cholesky_inv_banded(golden["cib_L"], 3), golden["cib_Pinv"], rtol=1e-12, atol=1e-14)


def test_melcd_oracle(golden):
    x, y = golden["melcd_x"], golden["melcd_y"]
    rows = np.array([oracle.cost(a, b, "melcd") for a, b in zip(x, y)])
    assert np.array_equal(rows, golden["melcd_rows"])  # bit-exact incl. numpy's pairwise summation order
    assert oracle.melcd(x, y) == float(golden["melcd_2d"])
    assert oracle.melcd(x[None], y[None], lengths=[4]) == float(golden["melcd_len"])
    assert oracle.melcd(x, x) == 0.0  # tests/test_metrics.py:8-32


def test_mlpg_oracle_edge_cases():
    ws = windows_set()[2]
    rng = np.random.default_rng(0)
    # T <= 2 * max_win_width: every dynamic precision is zeroed -> y == static mean
    for T in (1, 2):
        m = rng.random((T, 6))
        v = rng.random((T, 6)) + 0.1
        assert np.allclose(oracle.mlpg(m, v, ws), m[:, :2], rtol=1e-14)
    # D not a multiple of num_windows: static_dim = D // nw, trailing columns ignored (_mlpg.py:172)
    m = rng.random((9, 7)); v = rng.random((9, 7)) + 0.1
    assert oracle.mlpg(m, v, ws).shape == (9, 2)
    # non-positive pivot -> LinAlgError
    v2 = v.copy(); v2[:, 0] = -1.0
    with pytest.raises(np.linalg.LinAlgError):
        oracle.mlpg(m, v2, ws)


def test_oracle_vs_live_reference(parity_golden):
    # the reference's paramgen outputs on these inputs, stored by tests/golden/make_golden.py
    for wi, ws in enumerate(windows_set()):
        for dt in ("float32", "float64"):
            for T in (3, 17, 64):
                key = "live_w%d_%s_T%d" % (wi, dt, T)
                m, v, go = parity_golden[key + "_means"], parity_golden[key + "_vars"], parity_golden[key + "_go"]
                assert m.dtype == dt and m.shape == (T, 3 * len(ws))
                assert np.array_equal(parity_golden[key + "_y"], oracle.mlpg(m, v, ws)), key
                assert rel_err(oracle.mlpg_grad(m, v, ws, go), parity_golden[key + "_grad"]) < 2e-6, key
        R = parity_golden["live_w%d_R_T21" % wi]
        assert np.abs(R - oracle.unit_variance_mlpg_matrix(ws, 21)).max() < 1e-7


def test_delta_features_oracle(golden):
    # SURVEY section 8f row 2: preprocessing.delta_features, golden straight from the reference
    for wi, ws in enumerate(windows_set()):
        for dt in ("float32", "float64"):
            x = golden["delta_w%d_%s_x" % (wi, dt)]
            y = oracle.delta_features(x, ws)
            assert y.dtype == x.dtype and np.array_equal(y, golden["delta_w%d_%s_y" % (wi, dt)])
    # plain-array windows (non-bandmat form, generic.py:283-287)
    x = np.random.default_rng(0).random((7, 2))
    assert np.array_equal(oracle.delta_features(x, [np.array([1.0]), np.array([-0.5, 0.0, 0.5])]),
                          oracle.delta_features(x, windows_set()[1]))
