# -*- coding: utf-8 -*-
"""HODLR parity: CUDA path (through the C ABI) vs the CPU oracle and vs dense linear algebra.

Tolerances.  Tree / index structure: bit-exact.  Pivot sequences: exact in the cases listed (same RNG stream, argmax
not at a rounding knife-edge).  log-det / solve / log-likelihood: 1e-6 relative is the north-star bar; at tol=1e-10
both sides agree with the dense answer far better than that and we assert 1e-8.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _setup_solver_test(n=300, seed=1234):
    # reference tests/test_solvers.py:29-38
    from george_b200 import kernels as K
    np.random.seed(seed)
    x = np.sort(10 * np.random.randn(n))
    yerr = np.ones(n)
    kernel = 1.0 * K.ExpSquaredKernel(1.0)
    return kernel, x[:, None].copy(), yerr


def _structure(nodes):
    keys = ("start", "size", "half", "is_leaf", "parent", "direction", "depth")
    return [tuple(nd[k] for k in keys) for nd in nodes]


def test_reference_solver_case_and_pivots(gpu, oracle):
    """tests/test_solvers.py:29-62 (HODLR at tol=1e-10) + SURVEY.md App. B golden pivots."""
    from george_b200.solvers._hodlr import HODLRSolver
    from george_b200._spec import flatten
    kernel, x, yerr = _setup_solver_test()
    spec = flatten(kernel)
    K = oracle.value_symmetric(spec, x) + np.diag(yerr ** 2)
    for mode in ("reference", "pernode"):
        s = HODLRSolver()
        s.compute(kernel, x, yerr, min_size=100, tol=1e-10, seed=42, rng_mode=mode)
        assert s.computed
        o = oracle.HODLR(spec, x, yerr, min_size=100, tol=1e-10, seed=42, rng_mode=1 if mode == "reference" else 0)
        assert _structure(s.nodes()) == _structure(o.nodes())
        root = s.nodes()[0]
        assert root["rank"] == 14 and root["rng_draws"] == 33 and root["dense_fallback"] == 0
        rows, cols = s.pivots(0, 14)
        assert list(rows) == [56, 26, 86, 22, 62, 21, 13, 8, 45, 19, 2, 7, 0, 35]
        assert list(cols) == [149, 148, 144, 135, 146, 131, 124, 140, 118, 133, 112, 145, 106, 127]
        sign, ld = np.linalg.slogdet(K)
        assert np.allclose(s.log_determinant, ld)
        assert abs(s.log_determinant - 69.730382271778) < 1e-9
        assert abs(s.log_determinant - o.log_determinant) < 1e-9
        y = np.sin(x[:, 0])
        b = s.apply_inverse(y)
        assert b.shape == (300, 1)
        assert np.allclose(b[:, 0], np.linalg.solve(K, y))
        np.testing.assert_allclose(b[:, 0], o.apply_inverse(y), rtol=1e-8, atol=1e-10)
        assert np.allclose(s.apply_inverse(K), np.eye(300))
        assert np.allclose(s.get_inverse(), np.linalg.inv(K))
        assert abs(s.dot_solve(y) - y @ np.linalg.solve(K, y)) < 1e-8


@pytest.mark.parametrize("n,min_size", [(50, 100), (199, 100), (200, 100), (201, 100), (777, 50), (2000, 100),
                                         (4097, 64)])
def test_tree_structure_bit_exact(gpu, oracle, n, min_size):
    from george_b200 import kernels as K
    from george_b200.solvers._hodlr import HODLRSolver
    from george_b200._spec import flatten
    rng = np.random.default_rng(3)
    x = np.sort(rng.uniform(0, 10 * n / 1000, n))[:, None]
    yerr = 0.1 * np.ones(n)
    kernel = 1.0 * K.ExpSquaredKernel(1.0)
    s = HODLRSolver()
    s.compute(kernel, x, yerr, min_size=min_size, tol=1e-10, seed=42)
    o = oracle.HODLR(flatten(kernel), x, yerr, min_size=min_size, tol=1e-10, seed=42, rng_mode=0)
    assert _structure(s.nodes()) == _structure(o.nodes())
    assert abs(s.log_determinant - o.log_determinant) <= 1e-8 * abs(o.log_determinant)


@pytest.mark.parametrize("mode", ["pernode", "reference"])
@pytest.mark.parametrize("kname", ["expsq", "m32", "cfg5", "m52_3d"])
def test_values_vs_oracle_and_dense(gpu, oracle, mode, kname):
    from george_b200 import kernels as K
    from george_b200.solvers._hodlr import HODLRSolver
    from george_b200._spec import flatten
    rng = np.random.default_rng(5)
    n = 1500
    if kname == "m52_3d":
        x = rng.uniform(0, 1, (n, 3))
        x = x[np.argsort(x[:, 0])]
        kernel = 1.0 * K.Matern52Kernel(0.5, ndim=3)
        tol = 1e-12
    else:
        x = np.sort(rng.uniform(0, 10 * n / 1000, n))[:, None]
        kernel = {"expsq": 1.0 * K.ExpSquaredKernel(1.0), "m32": 1.0 * K.Matern32Kernel(1.0),
                  "cfg5": 1.0 * K.ExpSquaredKernel(1.0) + 0.5 * K.ExpSine2Kernel(gamma=1.0, log_period=np.log(3.0))}[kname]
        tol = 1e-10
    yerr = 0.1 * np.ones(n)
    y = np.sin(x[:, 0]) + 0.1 * rng.normal(size=n)
    spec = flatten(kernel)
    s = HODLRSolver()
    s.compute(kernel, x, yerr, min_size=100, tol=tol, seed=42, rng_mode=mode)
    o = oracle.HODLR(spec, x, yerr, min_size=100, tol=tol, seed=42, rng_mode=1 if mode == "reference" else 0)
    Kd = oracle.value_symmetric(spec, x) + np.diag(yerr ** 2)
    ld = np.linalg.slogdet(Kd)[1]
    assert abs(s.log_determinant - o.log_determinant) <= 1e-8 * abs(ld)
    assert abs(s.log_determinant - ld) <= 1e-7 * abs(ld)
    a = s.apply_inverse(y)[:, 0]
    ad = np.linalg.solve(Kd, y)
    assert np.linalg.norm(a - ad) <= 1e-6 * np.linalg.norm(ad)
    assert np.linalg.norm(a - o.apply_inverse(y)) <= 1e-6 * np.linalg.norm(ad)
    assert abs(s.dot_solve(y) - y @ ad) <= 1e-8 * abs(y @ ad)
    # ranks: identical to the oracle's when the pivot stream is the same (knife-edge free in these cases)
    gn, on = s.nodes(), o.nodes()
    if kname in ("expsq", "cfg5"):
        assert [nd["rank"] for nd in gn] == [nd["rank"] for nd in on]
        assert [nd["rng_draws"] for nd in gn] == [nd["rng_draws"] for nd in on]
    else:
        # m32 is exactly rank 2 in 1-D, so whether a rounding-noise pivot >= 1e-14 is found (rank 3) or the rows run out
        # (dense fallback, hodlr.h:161-176) depends on the last bits of exp(); m52_3d at tol=1e-12 converges at the
        # noise floor.  Value parity above is the contract; ranks may differ by noise.
        assert [nd["is_leaf"] for nd in gn] == [nd["is_leaf"] for nd in on]


def test_default_tolerance_matches_oracle_pivots(gpu, oracle):
    """At the default tol=0.1 the HODLR answer is NOT the dense answer (SURVEY.md App. A); parity with the reference
    then means reproducing its pivots, which rng_mode='reference' does."""
    from george_b200 import kernels as K
    from george_b200.solvers._hodlr import HODLRSolver
    from george_b200._spec import flatten
    rng = np.random.default_rng(9)
    n = 2000
    x = np.sort(rng.uniform(0, 10 * n / 1000, n))[:, None]
    yerr = 0.1 * np.ones(n)
    y = np.sin(x[:, 0])
    kernel = 1.0 * K.ExpSquaredKernel(1.0)
    s = HODLRSolver()
    s.compute(kernel, x, yerr, rng_mode="reference")  # defaults: min_size=100, tol=0.1, seed=42
    o = oracle.HODLR(flatten(kernel), x, yerr)
    for i, (a, b) in enumerate(zip(s.nodes(), o.nodes())):
        assert a["rank"] == b["rank"] and a["rng_draws"] == b["rng_draws"]
        if not a["is_leaf"]:
            ra, ca = s.pivots(i, a["rank"])
            rb, cb = o.pivots(i, b["rank"])
            assert list(ra) == list(rb) and list(ca) == list(cb)
    assert abs(s.log_determinant - o.log_determinant) <= 1e-9 * abs(o.log_determinant)
    assert abs(s.dot_solve(y) - o.dot_solve(y)) <= 1e-6 * abs(o.dot_solve(y))


def test_strange_hodlr_bug(gpu):
    """reference tests/test_solvers.py:64-75: must not crash at defaults."""
    import george_b200 as george
    from george_b200 import kernels
    np.random.seed(1234)
    x = np.sort(np.random.uniform(0, 10, 50000))
    yerr = 0.1 * np.ones_like(x)
    y = np.sin(x)
    kernel = np.var(y) * kernels.ExpSquaredKernel(1.0)
    gp_hodlr = george.GP(kernel, solver=george.HODLRSolver, seed=42)
    n = 200
    gp_hodlr.compute(x[:n], yerr[:n])
    gp_hodlr.log_likelihood(y[:n])


def test_sharded_compute_without_communicator_is_refused(gpu):
    """A sharded factorisation is collective: without the library's communicator it must fail up front, not return a
    handle that is uncomputed or holds one shard's partial log-determinant."""
    from george_b200.solvers._hodlr import HODLRSolver
    kernel, x, yerr = _setup_solver_test()
    s = HODLRSolver()
    with pytest.raises(ValueError, match="communicator"):
        s.compute(kernel, x, yerr, min_size=100, tol=1e-10, shard_rank=0, shard_count=2)
    assert s.computed == 0


def test_docs_golden_loglikelihood(gpu):
    """docs/tutorials/scaling.rst:56-91: log-likelihood 133.946394912 for both solvers at N=100."""
    import george_b200 as george
    from george_b200 import kernels
    np.random.seed(1234)
    x = np.sort(np.random.uniform(0, 10, 50000))
    yerr = 0.1 * np.ones_like(x)
    y = np.sin(x)
    kernel = np.var(y) * kernels.ExpSquaredKernel(1.0)
    for solver in (george.BasicSolver, george.HODLRSolver):
        gp = george.GP(kernel, solver=solver)
        gp.compute(x[:100], yerr[:100])
        assert abs(gp.log_likelihood(y[:100]) - 133.946394912) < 1e-6


def test_exhaust_lowrank_matches_dense_mode(gpu, oracle):
    """Matern-3/2 is exactly rank 2 on sorted 1-D inputs: most nodes run out of candidate rows.  The reference then
    stores the block densely (hodlr.h:161-176, exhaust='dense'); exhaust='lowrank' keeps the verified factors.  Both must
    give the reference's answer; the second must do it with rank <= 3 everywhere."""
    from george_b200 import kernels as K
    from george_b200.solvers._hodlr import HODLRSolver
    from george_b200._spec import flatten
    rng = np.random.default_rng(12)
    n = 3000
    x = np.sort(rng.uniform(0, 10 * n / 1000, n))[:, None]
    yerr = 0.1 * np.ones(n)
    y = np.sin(x[:, 0]) + 0.1 * rng.normal(size=n)
    kernel = 1.0 * K.Matern32Kernel(1.0)
    o = oracle.HODLR(flatten(kernel), x, yerr, min_size=100, tol=1e-10, seed=42, rng_mode=0)
    assert any(nd["dense_fallback"] for nd in o.nodes())  # the hazard is real for the reference algorithm
    res = {}
    for mode in ("dense", "lowrank"):
        s = HODLRSolver()
        s.compute(kernel, x, yerr, min_size=100, tol=1e-10, seed=42, exhaust=mode)
        res[mode] = (s.log_determinant, s.dot_solve(y), s.nodes())
    for mode in res:
        assert abs(res[mode][0] - o.log_determinant) <= 1e-10 * abs(o.log_determinant)
        assert abs(res[mode][1] - o.dot_solve(y)) <= 1e-8 * abs(o.dot_solve(y))
    assert max(nd["rank"] for nd in res["lowrank"][2]) <= 3
    assert any(nd["dense_fallback"] for nd in res["lowrank"][2])   # the flag still reports the exhausted nodes
    assert max(nd["rank"] for nd in res["dense"][2]) >= 100         # reference semantics: rank = min(rows, cols)


def _pivot_lists(s, nodes):
    out = []
    for i, nd in enumerate(nodes):
        if nd["is_leaf"]:
            out.append(None)
        else:
            r, c = s.pivots(i, nd["rank"])
            out.append((list(r), list(c)))
    return out


@pytest.mark.parametrize("kname,n,min_size", [("m32", 6000, 100), ("m32", 20000, 256), ("expsq", 20000, 100),
                                               ("m52", 9000, 100), ("exp", 5000, 64), ("prod_expsq_es2", 12000, 100)])
def test_bound_culling_is_decision_exact(gpu, monkeypatch, kname, n, min_size):
    """a2_eval skips (candidate row, 128-column group) pairs whose residual is PROVABLY < 1e-14 (kernel bound at the gap
    + |U| * max|V|).  That must not change a single decision: ranks, RNG draws, exhausted flags and pivot lists are
    identical to the exhaustive scan (BGP_NO_CULL=1); the scalars agree to the last bits (the up-sweep's split-K Gram
    products use floating-point atomics, so two runs of the SAME configuration already differ by an ulp or two)."""
    from george_b200 import kernels as K
    from george_b200.solvers._hodlr import HODLRSolver
    rng = np.random.default_rng(21)
    x = np.sort(rng.uniform(0, 10 * n / 1000, n))[:, None]
    yerr = 0.1 * np.ones(n)
    y = np.sin(x[:, 0]) + 0.1 * rng.normal(size=n)
    kernel = {"m32": 1.0 * K.Matern32Kernel(1.0), "expsq": 1.5 * K.ExpSquaredKernel(2.0), "m52": K.Matern52Kernel(0.7),
              "exp": 0.8 * K.ExpKernel(1.0),
              "prod_expsq_es2": 1.2 * K.ExpSquaredKernel(50.0) * K.ExpSine2Kernel(gamma=1.0, log_period=np.log(3.0))}[kname]
    res = {}
    for cull in (True, False):
        if cull:
            monkeypatch.delenv("BGP_NO_CULL", raising=False)
        else:
            monkeypatch.setenv("BGP_NO_CULL", "1")
        s = HODLRSolver()
        s.compute(kernel, x, yerr, min_size=min_size, tol=1e-10, seed=42, exhaust="lowrank")
        nodes = s.nodes()
        prof = s.aca_profile()
        res[cull] = (s.log_determinant, s.dot_solve(y), [(nd["rank"], nd["rng_draws"], nd["dense_fallback"]) for nd in nodes],
                     _pivot_lists(s, nodes), prof)
    monkeypatch.delenv("BGP_NO_CULL", raising=False)
    assert res[True][2] == res[False][2]
    assert res[True][3] == res[False][3]
    assert abs(res[True][0] - res[False][0]) <= 1e-13 * abs(res[False][0])
    assert abs(res[True][1] - res[False][1]) <= 1e-12 * abs(res[False][1])
    # the culled run verified the same number of entries and evaluated no more than the exhaustive one (which evaluates
    # every entry of every speculative candidate row: at least the verified ones)
    assert res[True][4]["evals"] == res[False][4]["evals"]
    assert res[True][4]["evaluated"] <= res[False][4]["evaluated"]
    assert res[False][4]["evaluated"] >= res[False][4]["evals"]


@pytest.mark.parametrize("kname", ["expsq", "sum_expsq_es2", "prod_expsq_es2", "sum_m32_es2", "prod_m32_es2", "m32"])
def test_lowrank_mode_matches_oracle_lowrank(gpu, oracle, kname):
    """exhaust='lowrank' + per-node RNG streams, the mode the headline runs in, against the oracle restated in the SAME
    mode (oracle.HODLR(rng_mode=0, exhaust=1)): structure, ranks, draws, pivots and scalars.  The specialised two-term
    evaluators (c*A + c2*ExpSine2, (c*A)*ExpSine2) are exercised here too: they must take the interpreter's decisions."""
    from george_b200 import kernels as K
    from george_b200.solvers._hodlr import HODLRSolver
    from george_b200._spec import flatten
    rng = np.random.default_rng(33)
    n = 2500
    x = np.sort(rng.uniform(0, 10 * n / 1000, n))[:, None]
    yerr = 0.1 * np.ones(n)
    y = np.sin(x[:, 0]) + 0.1 * rng.normal(size=n)
    es2 = K.ExpSine2Kernel(gamma=1.0, log_period=np.log(3.0))
    kernel = {"expsq": 1.0 * K.ExpSquaredKernel(1.0), "m32": 1.0 * K.Matern32Kernel(1.0),
              "sum_expsq_es2": 1.0 * K.ExpSquaredKernel(1.0) + 0.5 * es2,
              "prod_expsq_es2": 1.3 * K.ExpSquaredKernel(30.0) * es2,
              "sum_m32_es2": 0.7 * K.Matern32Kernel(2.0) + es2,
              "prod_m32_es2": K.Matern32Kernel(40.0) * es2}[kname]
    s = HODLRSolver()
    s.compute(kernel, x, yerr, min_size=100, tol=1e-10, seed=42, exhaust="lowrank")
    o = oracle.HODLR(flatten(kernel), x, yerr, min_size=100, tol=1e-10, seed=42, rng_mode=0, exhaust=1)
    gn, on = s.nodes(), o.nodes()
    assert _structure(gn) == _structure(on)
    assert abs(s.log_determinant - o.log_determinant) <= 1e-9 * abs(o.log_determinant)
    assert abs(s.dot_solve(y) - o.dot_solve(y)) <= 1e-7 * abs(o.dot_solve(y))
    if kname != "m32":
        # The pivot sequence is reproduced while the residual is above the rounding noise.  The LAST pivots of a node at
        # tol = 1e-10 are chosen among residual entries of 1e-13 .. 1e-15 (at the 1e-14 rejection threshold of
        # hodlr.h:191), where a fused multiply-add (device) against a separate multiply and add (the oracle, x86-64
        # baseline) decides: the first half of every node's pivot list must be identical, the rank within 25 %.
        for i, nd in enumerate(gn):
            if not nd["is_leaf"]:
                ra, ca = s.pivots(i, nd["rank"])
                rb, cb = o.pivots(i, on[i]["rank"])
                half = min(nd["rank"], on[i]["rank"]) // 2
                assert list(ra[:half]) == list(rb[:half]) and list(ca[:half]) == list(cb[:half]), i
                assert abs(nd["rank"] - on[i]["rank"]) <= max(2, on[i]["rank"] // 4), i
                assert nd["dense_fallback"] == on[i]["dense_fallback"]
    else:  # m32: exactly rank 2, the third pivot is rounding noise of exp() (see test_values_vs_oracle_and_dense)
        assert max(nd["rank"] for nd in gn) <= 3


def test_get_inverse_orientation_at_loose_tolerance(gpu, oracle):
    """get_inverse() must return M with M[:, j] = solve(e_j), the orientation of the reference's Eigen -> numpy
    conversion (_hodlr.cpp:193-199).  (The HODLR approximation is itself symmetric — K12 = K21^T by construction,
    hodlr.h:54-55 — so M differs from its transpose only by the rounding of the pivoted LU solves.)"""
    from george_b200 import kernels as K
    from george_b200.solvers._hodlr import HODLRSolver
    rng = np.random.default_rng(4)
    n = 700
    x = np.sort(rng.uniform(0, 7, n))[:, None]
    s = HODLRSolver()
    s.compute(1.0 * K.ExpSquaredKernel(1.0), x, 0.1 * np.ones(n), rng_mode="reference")  # tol = 0.1
    M = s.get_inverse()
    e = np.zeros(n)
    for j in (0, 123, 350, 699):
        e[:] = 0.0
        e[j] = 1.0
        np.testing.assert_allclose(M[:, j], s.apply_inverse(e)[:, 0], rtol=0, atol=1e-12 * np.abs(M).max())


def test_graph_loop_equals_host_driven_loop(gpu, monkeypatch):
    """The lock-step ACA loop runs as ONE CUDA-graph launch (a WHILE node fed by a2_tick_kernel) unless BGP_NO_GRAPH is
    set or per-kernel profiling is on; the two drivers must produce the same factorisation."""
    from george_b200 import kernels as K
    from george_b200.solvers._hodlr import HODLRSolver
    rng = np.random.default_rng(7)
    n = 9000
    x = np.sort(rng.uniform(0, 10 * n / 1000, n))[:, None]
    yerr = 0.1 * np.ones(n)
    y = np.sin(x[:, 0]) + 0.1 * rng.normal(size=n)
    res = {}
    for kname, kernel, exhaust in (("expsq", 1.0 * K.ExpSquaredKernel(1.0), "dense"), ("m32", 1.0 * K.Matern32Kernel(1.0), "lowrank")):
        for graph in (True, False):
            if graph:
                monkeypatch.delenv("BGP_NO_GRAPH", raising=False)
            else:
                monkeypatch.setenv("BGP_NO_GRAPH", "1")
            s = HODLRSolver()
            for _ in range(2):  # second compute: cached executable graph, warm capacities
                s.compute(kernel, x, yerr, min_size=100, tol=1e-10, seed=42, exhaust=exhaust)
            nodes = s.nodes()
            res[graph] = (s.log_determinant, s.dot_solve(y), [(nd["rank"], nd["rng_draws"], nd["dense_fallback"]) for nd in nodes],
                          _pivot_lists(s, nodes))
        monkeypatch.delenv("BGP_NO_GRAPH", raising=False)
        assert res[True][2] == res[False][2] and res[True][3] == res[False][3], kname
        assert abs(res[True][0] - res[False][0]) <= 1e-13 * abs(res[False][0])
        assert abs(res[True][1] - res[False][1]) <= 1e-12 * abs(res[False][1])


@pytest.mark.parametrize("kname", ["expsq", "m52", "sum"])
def test_plugin_defaults_return_the_reference_answer(gpu, oracle, kname):
    """A user who switches from george to this package and changes NOTHING (HODLRSolver defaults: min_size=100, tol=0.1,
    seed=42) must get george's number.  At tol = 0.1 the HODLR answer is not the dense answer (SURVEY.md App. A), so
    this requires the reference's pivot order: the plug-in resolves rng_mode=None to the reference stream for
    tol > 1e-6 (and to the level-parallel per-node streams for tight tolerances)."""
    import george_b200 as george
    from george_b200 import kernels as K
    from george_b200._spec import flatten
    from george_b200.solvers._hodlr import resolve_rng_mode
    assert resolve_rng_mode(None, 0.1) == "reference" and resolve_rng_mode(None, 1e-10) == "pernode"
    assert resolve_rng_mode("pernode", 0.1) == "pernode"
    rng = np.random.default_rng(17)
    n = 3000
    x = np.sort(rng.uniform(0, 10 * n / 1000, n))
    yerr = 0.1 * np.ones(n)
    y = np.sin(x) + 0.1 * rng.normal(size=n)
    kernel = {"expsq": np.var(y) * K.ExpSquaredKernel(1.0), "m52": 1.0 * K.Matern52Kernel(2.0),
              "sum": 1.0 * K.ExpSquaredKernel(1.0) + 0.5 * K.ExpSine2Kernel(gamma=1.0, log_period=np.log(3.0))}[kname]
    gp = george.GP(kernel, solver=george.HODLRSolver)   # all defaults
    gp.compute(x, yerr)
    ll = gp.log_likelihood(y)
    sigma = np.sqrt(yerr ** 2 + george.gp.TINY)
    o = oracle.HODLR(flatten(kernel), x, sigma)         # the restated reference at ITS defaults (shared rng, dense fallback)
    ll_ref = -0.5 * (n * np.log(2 * np.pi) + o.log_determinant) - 0.5 * o.dot_solve(y)
    assert abs(ll - ll_ref) <= 1e-6 * abs(ll_ref)
    # ... and it is NOT what the per-node streams give at this tolerance (which is why the default matters)
    gp2 = george.GP(kernel, solver=george.HODLRSolver, rng_mode="pernode")
    gp2.compute(x, yerr)
    assert np.isfinite(gp2.log_likelihood(y))


def test_ill_conditioned_system_matches_oracle(gpu, oracle):
    """Smooth kernel, small noise: cond(K) ~ 1e7, leaf pivots D down to 1e-4 and Woodbury matrices S with pivots spread over
    several decades (at cond 1e11 the reference algorithm itself loses the log-det to 1e-3: nothing to compare there).  The reference factors leaves with Eigen's pivoted LDLT and S with FullPivLU (hodlr.h:23-24,227,233);
    the device uses un-pivoted LDL^T (equal for SPD leaves up to rounding) and complete-pivoting LU with FullPivLU's
    rank threshold.  log-det and solve must agree with the oracle at the level the conditioning allows."""
    from george_b200 import kernels as K
    from george_b200.solvers._hodlr import HODLRSolver
    from george_b200._spec import flatten
    rng = np.random.default_rng(2)
    n = 1200
    x = np.sort(rng.uniform(0, 12, n))[:, None]
    yerr = 1e-2 * np.ones(n)
    y = np.sin(x[:, 0])
    kernel = 1.0 * K.ExpSquaredKernel(25.0)
    for mode in ("reference", "pernode"):
        s = HODLRSolver()
        s.compute(kernel, x, yerr, min_size=100, tol=1e-12, seed=42, rng_mode=mode)
        o = oracle.HODLR(flatten(kernel), x, yerr, min_size=100, tol=1e-12, seed=42, rng_mode=1 if mode == "reference" else 0)
        assert np.isfinite(s.log_determinant)
        assert abs(s.log_determinant - o.log_determinant) <= 1e-9 * abs(o.log_determinant)
        a, ao = s.apply_inverse(y)[:, 0], o.apply_inverse(y)
        assert np.linalg.norm(a - ao) <= 1e-6 * np.linalg.norm(ao)     # cond * eps ~ 1e-9 on each side
        Kd = oracle.value_symmetric(flatten(kernel), x) + np.diag(yerr ** 2)
        assert np.linalg.norm(Kd @ a - y) <= 1e-7 * np.linalg.norm(y)


def test_rank_deficient_woodbury_matrix_is_truncated_like_fullpivlu(gpu, oracle):
    """Two identical points, one in each half of the root, and NO noise: the leaves are regular but K is exactly singular,
    so the root's 2r x 2r Woodbury matrix S is rank deficient.  Eigen::FullPivLU::solve (hodlr.h:250) drops the pivots
    below eps * n * |max pivot| (a pseudo-solve) instead of dividing by rounding noise; the device LU follows the same
    rule, so the solve stays finite and agrees with the restated reference."""
    from george_b200 import kernels as K
    from george_b200.solvers._hodlr import HODLRSolver
    from george_b200._spec import flatten
    rng = np.random.default_rng(8)
    n = 140
    x = np.sort(rng.uniform(0, 4, n))
    x[100] = x[30]                       # same point in the left (0..69) and the right (70..139) leaf
    x = x[:, None]
    yerr = np.zeros(n)
    y = np.sin(x[:, 0])
    kernel = 1.0 * K.ExpKernel(0.25)     # rough kernel: the two leaves are well conditioned (cond ~ 1e5) without noise;
    # exp(-|d|) is exactly rank 1 between sorted halves, so the root exhausts its rows and stores the block densely
    # (hodlr.h:161-176): r = 70 and S is 140 x 140 with ONE vanishing pivot
    s = HODLRSolver()
    s.compute(kernel, x, yerr, min_size=70, tol=1e-12, seed=42, rng_mode="reference")
    o = oracle.HODLR(flatten(kernel), x, yerr, min_size=70, tol=1e-12, seed=42, rng_mode=1)
    assert s.nodes()[0]["rank"] == 70 and o.nodes()[0]["rank"] == 70
    a, ao = s.apply_inverse(y)[:, 0], o.apply_inverse(y)
    assert np.all(np.isfinite(a)) and np.all(np.isfinite(ao))
    scale = np.linalg.norm(ao)
    assert scale < 1e8                   # truncated: a division by the noise pivot would give ~1e15
    assert np.linalg.norm(a - ao) <= 1e-4 * scale
