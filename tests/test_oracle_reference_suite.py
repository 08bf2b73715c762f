"""Pins the CPU oracle against every test the reference's own suite holds for this path
(staple/spark-agd's src/test/scala/.../AcceleratedGradientDescentSuite.scala, cited as Suite.scala)
and against the one Java known-answer value available (java.util.Random(42).nextGaussian()).

The reference ships no golden vectors; tests/golden/reference_suite_anchors.json holds the values
this oracle produced when it was first checked against SURVEY.md 8(c)'s independent numpy
restatement -- a regression anchor, not a reference-emitted golden."""
import json
import os

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


def rel_close(a, b, eps):
    """TestingUtils `~= relTol`: |a-b| < eps * min(|a|,|b|) [mllib-1.3.0 tests]."""
    return abs(a - b) < eps * min(abs(a), abs(b))


def test_java_random_known_answers(oracle):
    # new java.util.Random(42).nextGaussian() is the well-known 1.1419053154730547
    x1, _ = oracle.generate_gd_input(2.0, -1.5, 4, 42)
    assert x1[0] == 1.1419053154730547
    # new java.util.Random(0).nextDouble() = 0.730967787376657
    assert oracle.jrandom_doubles(0, 1)[0] == 0.730967787376657
    # new java.util.Random(42).nextDouble() = 0.7275636800328681
    assert oracle.jrandom_doubles(42, 1)[0] == 0.7275636800328681


def test_fixture_shape(oracle, fixture_gd_input):
    y, X = fixture_gd_input
    assert X.shape == (10000, 2) and set(np.unique(y)) == {0.0, 1.0}
    assert abs(y.mean() - 0.8133) < 1e-12


def test_T1_unregularised_loss_matches_gd(oracle, fixture_gd_input):          # Suite.scala:53-91
    y, X = fixture_gd_input
    D = oracle.Data(y, X=X)
    r = oracle.agd_run(D, "logistic", "simple", [1.0, -1.0], convergence_tol=1e-12, num_iterations=10,
                       reg_param=0.0, L0=1.0, Lexact=float("inf"), beta=0.5, alpha=0.9, may_restart=True)
    _, loss_gd = oracle.gd_run(D, "logistic", "simple", [1.0, -1.0], step_size=1.0, num_iterations=50)
    assert rel_close(r.loss_history[-1], loss_gd[-1], 0.02)
    assert r.passes == 30 and r.backtracks == 0           # exactly 3 applySmooth per iteration


def test_T2_l2_regularised(oracle, fixture_gd_input):                         # Suite.scala:93-136
    y, X = fixture_gd_input
    D = oracle.Data(y, X=X)
    r = oracle.agd_run(D, "logistic", "squared_l2", [0.3, 0.12], convergence_tol=1e-12, num_iterations=10,
                       reg_param=0.2)
    w_gd, loss_gd = oracle.gd_run(D, "logistic", "squared_l2", [0.3, 0.12], step_size=1.0, num_iterations=50,
                                  reg_param=0.2)
    assert rel_close(r.loss_history[-1], loss_gd[-1], 0.02)
    assert rel_close(r.weights[0], w_gd[0], 0.02) and rel_close(r.weights[1], w_gd[1], 0.02)


def test_T3_convergence_tol(oracle, fixture_gd_input):                        # Suite.scala:138-207
    y, X = fixture_gd_input
    D = oracle.Data(y, X=X)
    r1 = oracle.agd_run(D, "logistic", "squared_l2", [0.0, 0.0], convergence_tol=0.1, num_iterations=1000)
    r2 = oracle.agd_run(D, "logistic", "squared_l2", [0.0, 0.0], convergence_tol=0.0,
                        num_iterations=len(r1.loss_history) - 1)
    assert len(r2.loss_history) == len(r1.loss_history) - 1
    assert np.linalg.norm(r1.weights - r2.weights) / np.linalg.norm(r1.weights) < 0.1
    r3 = oracle.agd_run(D, "logistic", "squared_l2", [0.0, 0.0], convergence_tol=0.01, num_iterations=100)
    assert len(r3.loss_history) > len(r1.loss_history)


def test_T4_class_defaults(oracle, fixture_gd_input):                         # Suite.scala:209-239
    y, X = fixture_gd_input
    D = oracle.Data(y, X=X)
    r = oracle.agd_run(D, "logistic", "squared_l2", [1.0, -1.0], convergence_tol=1e-12, num_iterations=10,
                       reg_param=0.2)
    w_gd, _ = oracle.gd_run(D, "logistic", "squared_l2", [1.0, -1.0], step_size=1.0, num_iterations=50, reg_param=0.2)
    assert rel_close(r.weights[0], w_gd[0], 0.02) and rel_close(r.weights[1], w_gd[1], 0.02)


def test_T5_wide_rows_one_iteration(oracle):                                  # Suite.scala:244-259
    m, n = 10, 200000  # the suite's own size (it exists to trip Spark's 1 MB frame size with 10 x 200000 doubles)
    rows = [oracle.jrandom_doubles(idx, (m // 2) * n).reshape(m // 2, n) for idx in (0, 1)]
    X = np.concatenate(rows, axis=0)
    y = np.ones(m)
    w0 = oracle.jrandom_doubles(0, n)
    r = oracle.agd_run(oracle.Data(y, X=X), "logistic", "squared_l2", w0, convergence_tol=1e-12, num_iterations=1,
                       reg_param=1.0)
    assert len(r.loss_history) == 1 and np.all(np.isfinite(r.weights))


def test_anchor_values(oracle, fixture_gd_input):
    y, X = fixture_gd_input
    D = oracle.Data(y, X=X)
    with open(os.path.join(HERE, "golden", "reference_suite_anchors.json")) as f:
        G = json.load(f)
    r = oracle.agd_run(D, "logistic", "simple", [1.0, -1.0], convergence_tol=1e-12, num_iterations=10)
    np.testing.assert_allclose(r.loss_history, G["T1_agd_loss_history"], rtol=1e-13)
    np.testing.assert_allclose(r.weights, G["T1_agd_weights"], rtol=1e-13)
    _, lg = oracle.gd_run(D, "logistic", "simple", [1.0, -1.0], step_size=1.0, num_iterations=50)
    np.testing.assert_allclose(lg[-1], G["T1_gd_last_loss"], rtol=1e-13)
    r2 = oracle.agd_run(D, "logistic", "squared_l2", [0.3, 0.12], convergence_tol=1e-12, num_iterations=10,
                        reg_param=0.2)
    np.testing.assert_allclose(r2.weights, G["T2_agd_weights"], rtol=1e-13)
    # SURVEY.md 8(c): values from an independent numpy restatement (8 significant digits quoted there)
    np.testing.assert_allclose(r.loss_history, [0.40895983, 0.39907627, 0.39061099, 0.3842363, 0.37970851,
                                                0.3765193, 0.37430618, 0.37287803, 0.37207889, 0.37172288],
                               rtol=2e-8)
    np.testing.assert_allclose(r.weights, [1.98081281, -1.43474202], rtol=1e-8)
    np.testing.assert_allclose(r2.weights, [0.72783272, -0.41126233], rtol=2e-8)


@pytest.mark.parametrize("grad", ["logistic", "least_squares", "hinge"])
@pytest.mark.parametrize("upd", ["simple", "squared_l2", "l1"])
def test_oracle_against_numpy_formulas(oracle, grad, upd):
    """The un-vendored mllib-1.3.0 formulas (SURVEY.md 8(a6)-(a9)) restated a second time in numpy."""
    rng = np.random.default_rng(7)
    n, d = 300, 17
    X = rng.standard_normal((n, d))
    y = (rng.random(n) > 0.4).astype(np.float64) if grad != "least_squares" else rng.standard_normal(n)
    w = rng.standard_normal(d) * 0.3
    loss, g, cnt = oracle.smooth(oracle.Data(y, X=X), grad, w, partitions=3)
    m = X @ w
    if grad == "logistic":
        mult = 1.0 / (1.0 + np.exp(-m)) - y
        l = np.where(y > 0, np.logaddexp(0, -m), np.logaddexp(0, -m) + m)
    elif grad == "least_squares":
        mult, l = 2 * (m - y), (m - y) ** 2
    else:
        s = 2 * y - 1
        act = 1.0 > s * m
        mult, l = np.where(act, -s, 0.0), np.where(act, 1 - s * m, 0.0)
    np.testing.assert_allclose(loss, l.mean(), rtol=1e-12)
    np.testing.assert_allclose(g, (X * mult[:, None]).mean(axis=0), rtol=1e-10, atol=1e-14)
    assert cnt == n
    step, reg = 0.37, 0.21
    rv, wn = oracle.prox(upd, w, g, step, reg)
    if upd == "simple":
        exp_w, exp_r = w - step * g, 0.0
    elif upd == "squared_l2":
        exp_w = w * (1 - step * reg) - step * g
        exp_r = 0.5 * reg * np.dot(exp_w, exp_w)
    else:
        u = w - step * g
        exp_w = np.sign(u) * np.maximum(0, np.abs(u) - reg * step)
        exp_r = reg * np.abs(exp_w).sum()
    np.testing.assert_allclose(wn, exp_w, rtol=1e-13, atol=1e-16)
    np.testing.assert_allclose(rv, exp_r, rtol=1e-13)


def test_empty_data_flags_nonterminating(oracle):
    """count = 0 => 0/0 = NaN loss (AGD.scala:207); the reference then never leaves its backtracking
    loop (NaN fails :281 forever); the oracle stops and says so."""
    D = oracle.Data(np.zeros(0), X=np.zeros((0, 3)))
    r = oracle.agd_run(D, "logistic", "simple", [0.1, 0.2, 0.3], num_iterations=5)
    assert r.nonterminating and r.stopped_nan and len(r.loss_history) == 1 and np.isnan(r.loss_history[0])
