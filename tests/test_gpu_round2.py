"""Round-2 device features, each against the oracle / numpy on the same inputs: selection fused into the
kernel epilogue, streamed (chunked) host batches, the device Philox candidate source, the STABLE path
policy of the refinement runs, and the ADVICE regressions."""
import ctypes as C
import warnings

import numpy as np
import pytest
from numpy.testing import assert_allclose
from sklearn.gaussian_process.kernels import Matern

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def bo():
    import bayesianoptimization_b200 as bo

    return bo


@pytest.fixture(scope="module")
def O():
    from oracle import gp_oracle

    return gp_oracle


def _synth(n, d, seed=0):
    rs = np.random.RandomState(seed)
    X = rs.uniform(size=(n, d))
    y = np.sin(X.sum(1)) + 0.1 * rs.randn(n)
    return X, y


def _gp(bo, X, y, ls=0.7, **kw):
    return bo.B200GaussianProcessRegressor(kernel=Matern(nu=2.5, length_scale=ls), alpha=1e-6, normalize_y=True,
                                           optimizer=None, **kw).fit(X, y)


def _np_select(ys, k):
    """np.argmin (first NaN wins) and stable argsort[:k] (NaN last) - the reference's selection."""
    return int(np.argmin(ys)), np.argsort(ys, kind="stable")[:k]


@pytest.mark.parametrize("precision", ["fp64", "fp32"])
@pytest.mark.parametrize("m,k", [(129, 5), (5000, 10), (148 * 128 * 3 + 77, 64), (40_000, 1)])
def test_fused_selection_equals_numpy_on_the_same_values(bo, monkeypatch, precision, m, k):
    """argmin/top-k from the running per-CTA lists + k-way merge == np.argmin / stable argsort of the values
    the same kernel writes when asked to materialise them (ties, many CTAs, k up to 64)."""
    monkeypatch.setenv("B200BO_SMALL_PATH", "0")  # tiled persistent kernel whatever m is
    X, y = _synth(300, 4, 1)
    gp = _gp(bo, X, y, precision=precision)
    f = bo.FusedAcquisition(bo._lib.ACQ_EI, gp, xi=0.01, y_max=float(y.max()))
    rs = np.random.RandomState(m)
    xt = rs.uniform(size=(m, 4))
    xt[m // 2] = xt[3]          # exact ties across tiles
    xt[m - 1] = xt[3]
    xt[7] = xt[m // 3]
    ys = f(xt)
    assert ys[m // 2] == ys[3] == ys[m - 1]
    idx, val, top = f.argmin_topk(xt, k)
    ri, rtop = _np_select(ys, k)
    assert idx == ri and val == ys[ri]
    assert list(top) == list(rtop)


def test_fused_selection_nan_semantics(bo, monkeypatch):
    """sigma = 0 and a = 0 gives EI = NaN (0/0): np.argmin returns the FIRST NaN, argsort puts NaNs last."""
    monkeypatch.setenv("B200BO_SMALL_PATH", "0")
    X, y = _synth(60, 2, 3)
    gp = bo.B200GaussianProcessRegressor(kernel=Matern(nu=2.5, length_scale=0.5), alpha=1e-10, normalize_y=False,
                                         optimizer=None).fit(X, y)
    rs = np.random.RandomState(0)
    xt = rs.uniform(size=(3000, 2))
    f = bo.FusedAcquisition(bo._lib.ACQ_EI, gp, xi=0.0, y_max=0.0)
    ys = f(xt)
    idx, val, top = f.argmin_topk(xt, 8)
    ri, rtop = _np_select(ys, 8)
    assert idx == ri and list(top) == list(rtop)
    # force NaNs: a training point with y_max = its own target and xi = 0 -> a = 0, sigma ~ 0
    xt2 = xt.copy()
    xt2[[1500, 17, 2900]] = X[[4, 9, 4]]
    mu, sd = gp.predict(xt2[[17]], return_std=True)
    f2 = bo.FusedAcquisition(bo._lib.ACQ_EI, gp, xi=0.0, y_max=float(mu[0]))
    ys2 = f2(xt2)
    idx2, val2, top2 = f2.argmin_topk(xt2, 8)
    ri2, rtop2 = _np_select(ys2, 8)
    assert idx2 == ri2 and list(top2) == list(rtop2)
    if np.isnan(ys2).any():
        assert np.isnan(val2) and idx2 == int(np.flatnonzero(np.isnan(ys2))[0])


@pytest.mark.parametrize("precision", ["fp64", "fp32"])
def test_streamed_host_batch_equals_single_launch(bo, monkeypatch, precision):
    """A host batch >= 2 chunks is uploaded in chunks on a copy stream while the previous chunk is evaluated;
    the per-CTA selection lists carry over between launches.  Result == the one-launch path (B200BO_CHUNKED=0),
    bit for bit."""
    X, y = _synth(256, 6, 2)
    gp = _gp(bo, X, y, precision=precision)
    f = bo.FusedAcquisition(bo._lib.ACQ_EI, gp, xi=0.01, y_max=float(y.max()))
    m = 2 * 8 * 128 * 148 + 12345  # > 2 chunks, ragged tail
    xt = np.random.RandomState(5).uniform(size=(m, 6))
    xt[m - 3] = xt[100]
    a = f.argmin_topk(xt, 10)
    monkeypatch.setenv("B200BO_CHUNKED", "0")
    b = f.argmin_topk(xt, 10)
    assert a[0] == b[0] and a[1] == b[1] and list(a[2]) == list(b[2])
    ys = f(xt)
    ri, rtop = _np_select(ys, 10)
    assert a[0] == ri and list(a[2]) == list(rtop)


@pytest.mark.parametrize("d", [1, 2, 5, 16, 33])
def test_philox_rows_match_oracle_bitwise(bo, O, d):
    from bayesianoptimization_b200 import _lib as B

    lo = np.linspace(-1.0, 0.5, d)
    hi = lo + np.linspace(0.5, 3.0, d)
    idx = np.array([0, 1, 2, 127, 128, 12345, 2**31 - 1, 2**31, 2**40 + 17], dtype=np.int64)
    out = np.empty((len(idx), d))
    B.check(B.lib().b200bo_philox_rows(0, 0x1234_5678_9ABC_DEF0, B.as_dp(lo), B.as_dp(hi), d,
                                       idx.ctypes.data_as(C.POINTER(C.c_int64)), len(idx), B.as_dp(out)))
    ref = O.philox_uniform(0x1234_5678_9ABC_DEF0, idx, d, lo, hi)
    assert np.array_equal(out, ref)


@pytest.mark.parametrize("precision,n,d", [("fp64", 300, 4), ("fp32", 512, 8), ("fp64", 64, 17)])
def test_throughput_mode_equals_host_evaluation_of_the_same_rows(bo, O, precision, n, d):
    """argmin_topk_philox (candidates generated inside the kernel) == argmin_topk on the oracle's
    regeneration of the same Philox rows; winners' coordinates come back bit-exact."""
    X, y = _synth(n, d, 4)
    gp = _gp(bo, X, y, precision=precision)
    f = bo.FusedAcquisition(bo._lib.ACQ_EI, gp, xi=0.01, y_max=float(y.max()))
    m, k, seed, base = 30_000, 7, 42, 1_000_000
    bounds = np.column_stack([np.zeros(d), np.ones(d)])
    bounds[0] = (0.25, 0.75)
    idx, val, bx, top, tx = f.argmin_topk_philox(seed, bounds, m, k, index_base=base)
    rows = O.philox_uniform(seed, base + np.arange(m), d, bounds[:, 0], bounds[:, 1])
    hi_, hv, htop = f.argmin_topk(rows, k)
    assert idx == base + hi_ and val == hv and list(top) == list(base + htop)
    assert np.array_equal(bx, rows[hi_]) and np.array_equal(tx, rows[htop])
    # small-batch kernels generate the same rows
    i2, v2, bx2, top2, tx2 = f.argmin_topk_philox(seed, bounds, 20, 3, index_base=base)
    h2 = f.argmin_topk(rows[:20], 3)
    assert i2 == base + h2[0] and v2 == h2[1] and list(top2) == list(base + h2[2])


@pytest.mark.parametrize("n,d", [(100, 4), (128, 6), (60, 9)])
def test_lockstep_refinement_bit_identical_to_sequential_small_n(bo, ref, monkeypatch, n, d):
    """ADVICE r1: at small N the objective batch (n_seeds rows) and the stencil batch (n_seeds*d rows) used to
    pick different kernels; with B200BO_PATH_STABLE the lockstep run and the plain sequential loop see the
    same bits."""
    X, y = _synth(n, d, 7)
    gp = _gp(bo, X, y, ls=0.6)
    a = bo.ExpectedImprovement(xi=0.01)
    a.y_max = float(y.max())
    f = a._get_acq(gp=gp)
    space = ref.target_space.TargetSpace(None, {f"x{i:02d}": (0.0, 1.0) for i in range(d)})
    seeds = np.random.RandomState(1).uniform(size=(10, d))
    x1, v1 = a._smart_minimize(f, space, seeds, np.random.RandomState(0))
    monkeypatch.setenv("B200BO_LOCKSTEP", "0")
    x2, v2 = a._smart_minimize(f, space, seeds, np.random.RandomState(0))
    assert np.array_equal(x1, x2) and v1 == v2
    # and the values of one row do not depend on the batch it arrives in while in refine mode
    with f.refine_mode():
        big = f(np.vstack([seeds] * 9))
        one = np.array([f(s)[0] for s in seeds])
    assert np.array_equal(big[:10], one)


def test_n_smart_beyond_device_topk_capacity(bo, ref):
    """ADVICE r1: the reference accepts any n_smart (np.argsort(ys)[:n]); beyond B200BO_MAX_TOPK the hook
    evaluates on the device and selects with numpy instead of raising."""
    X, y = _synth(50, 2, 1)
    gp = _gp(bo, X, y)
    a = bo.UpperConfidenceBound(kappa=2.0)
    f = a._get_acq(gp=gp)
    space = ref.target_space.TargetSpace(None, {"x": (0.0, 1.0), "y": (0.0, 1.0)})
    x_min, v, seeds = a._random_sample_minimize(f, space, np.random.RandomState(3), n_random=500, n_x_seeds=100)
    xt = space.random_sample(500, np.random.RandomState(3))
    ys = f(xt)
    assert np.array_equal(seeds, xt[np.argsort(ys)[:100]]) and v == ys.min()


def test_user_base_acq_override_is_honoured_and_params_read_at_call_time(bo, ref):
    """ADVICE r1: a subclass of a stock acquisition that overrides base_acq must not get the built-in device
    epilogue; kappa / xi / y_max are read when the closure is CALLED, as in the reference."""
    X, y = _synth(80, 3, 2)
    gp = _gp(bo, X, y)
    xt = np.random.RandomState(0).uniform(size=(200, 3))

    class Shifted(bo.UpperConfidenceBound):
        def base_acq(self, mean, std):
            return mean + self.kappa * std + 5.0

    stock = bo.UpperConfidenceBound(kappa=1.5)
    f = stock._get_acq(gp=gp)
    assert isinstance(f, bo.FusedAcquisition)
    g = Shifted(kappa=1.5)._get_acq(gp=gp)
    assert not isinstance(g, bo.FusedAcquisition)
    assert_allclose(g(xt), f(xt) - 5.0, rtol=1e-12)
    y0 = f(xt)
    stock.kappa = 0.0
    mu = gp.predict(xt)
    assert_allclose(f(xt), -mu, rtol=1e-10, atol=1e-12)
    assert not np.allclose(y0, f(xt))
    e = bo.ExpectedImprovement(xi=0.0)
    h = e._get_acq(gp=gp)
    with pytest.raises(ValueError, match="y_max"):
        h(xt)
    e.y_max = float(y.max())
    assert h(xt).shape == (200,)


def test_gphedge_vs_golden(bo, ref, golden):
    """GPHedge over device base acquisitions reproduces the reference run of oracle/make_golden.py
    (case_gphedge): gains, candidates, softmax draws and suggestions."""
    from bayes_opt.parameter import wrap_kernel

    g = golden("gphedge_small")

    def f(x, y):
        return -((x - 3) ** 2) - (y - 1) ** 2 + 0.3 * np.sin(3 * x)

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        space = ref.target_space.TargetSpace(f, {"x": (1, 4), "y": (0, 3.0)})
        for x, t in zip(g["X"], g["y"]):
            space.register(x, t)
        gp = bo.B200GaussianProcessRegressor(kernel=wrap_kernel(Matern(nu=2.5, length_scale=0.9), space.kernel_transform),
                                             alpha=1e-6, normalize_y=True, optimizer=None)
        hedge = bo.GPHedge([bo.UpperConfidenceBound(kappa=2.0), bo.ExpectedImprovement(xi=0.01),
                            bo.ProbabilityOfImprovement(xi=0.01)])
        rng = np.random.RandomState(13)
        for it in range(4):
            gp.fit(space.params, space.target)
            x = hedge.suggest(gp, space, n_random=3000, n_smart=3, fit_gp=False, random_state=rng)
            assert_allclose(hedge.gains, g["gains"][it], rtol=1e-5, atol=1e-7)
            assert_allclose(hedge.previous_candidates, g["candidates"][it], rtol=1e-4, atol=1e-5)
            assert_allclose(x, g["suggestions"][it], rtol=1e-4, atol=1e-5)
            space.probe(g["suggestions"][it])  # continue from the reference's trajectory
    assert rng.rand() == float(g["next_rand"])  # the RNG stream was consumed identically


def test_lazy_lml_value_and_2d_validation(bo):
    """ADVICE r1: optimizer=None leaves log_marginal_likelihood_value_ a float (computed on first access);
    1-D X is rejected like sklearn's validate_data does."""
    from sklearn.gaussian_process import GaussianProcessRegressor

    X, y = _synth(40, 2, 5)
    gp = _gp(bo, X, y)
    sk = GaussianProcessRegressor(kernel=Matern(nu=2.5, length_scale=0.7), alpha=1e-6, normalize_y=True,
                                  optimizer=None).fit(X, y)
    assert gp.log_marginal_likelihood_value_ == pytest.approx(sk.log_marginal_likelihood_value_, rel=1e-9)
    assert_allclose(gp.predict(X[:5]), sk.predict(X[:5]), rtol=1e-6)
    with pytest.raises(ValueError):
        gp.predict(X[0])
    with pytest.raises(ValueError):
        bo.B200GaussianProcessRegressor(kernel=Matern(nu=2.5), optimizer=None).fit(X[:, 0], y)


@pytest.mark.parametrize("n,d", [(129, 3), (700, 5), (2048, 16), (4096, 16)])
def test_lookahead_cholesky_and_tiled_gemm_vs_serial_and_sklearn(bo, monkeypatch, n, d):
    """Fit side, round 2: look-ahead Cholesky (diagonal chain on one stream, panel solve + trailing update on a
    second one, potrf_diag_kernel resolving the previous panel itself) with 128x128 pipelined DMMA tiles,
    against (a) the serial loop on 64x64 tiles of round 1 (B200BO_POTRF=serial, B200BO_GEMM=64): same factor to
    round-off, (b) itself: bit-identical on repetition (no race between the two streams), (c) LML + gradient of
    sklearn."""
    from sklearn.gaussian_process import GaussianProcessRegressor

    from bayesianoptimization_b200 import _lib as B

    X, y = _synth(n, d, 3)

    def run():
        gp = _gp(bo, X, y, ls=0.8)
        W = np.empty((n, n))
        B.check(B.lib().b200bo_gp_get(gp._handle().ptr, B.GET_LINV, B.as_dp(W), n * n))
        lml, grad = gp.log_marginal_likelihood(np.log([0.6]), eval_gradient=True)
        return gp.L_.copy(), W, gp.alpha_.copy(), lml, grad

    a = run()
    b = run()
    for u, v in zip(a, b):
        assert np.array_equal(u, v)  # deterministic whatever the stream interleaving
    monkeypatch.setenv("B200BO_POTRF", "serial")
    monkeypatch.setenv("B200BO_GEMM", "64")
    c = run()
    assert_allclose(a[0], c[0], rtol=1e-8, atol=1e-11)
    assert np.all(np.triu(a[0], 1) == 0)
    assert np.max(np.abs(a[1] @ a[0] - np.eye(n))) < 1e-6
    assert_allclose(a[2], c[2], rtol=1e-6)
    assert a[3] == pytest.approx(c[3], rel=1e-9) and a[4][0] == pytest.approx(c[4][0], rel=1e-6)
    if n <= 2048:
        sk = GaussianProcessRegressor(kernel=Matern(nu=2.5, length_scale=0.8), alpha=1e-6, normalize_y=True,
                                      optimizer=None).fit(X, y)
        l0, g0 = sk.log_marginal_likelihood(np.log([0.6]), eval_gradient=True)
        assert a[3] == pytest.approx(l0, rel=1e-8) and a[4][0] == pytest.approx(g0[0], rel=1e-5, abs=1e-6)
        assert_allclose(a[0], sk.L_, rtol=1e-7, atol=1e-10)


@pytest.mark.parametrize("tag", ["aniso_const", "rbf_iso"])
def test_tiled_lml_gradient_kernel_families(bo, tag):
    """lml_grad_tile_kernel (templated covariance, iso/aniso, optional ConstantKernel) against sklearn."""
    from sklearn.gaussian_process import GaussianProcessRegressor
    from sklearn.gaussian_process.kernels import RBF, ConstantKernel

    X, y = _synth(300, 4, 8)
    if tag == "aniso_const":
        k = ConstantKernel(1.7) * Matern(nu=1.5, length_scale=[0.5, 0.9, 1.3, 0.7])
        theta = np.log([2.0, 0.6, 0.8, 1.1, 0.9])
    else:
        k = RBF(length_scale=0.8)
        theta = np.log([0.5])
    gp = bo.B200GaussianProcessRegressor(kernel=k, alpha=1e-6, normalize_y=True, optimizer=None).fit(X, y)
    sk = GaussianProcessRegressor(kernel=k, alpha=1e-6, normalize_y=True, optimizer=None).fit(X, y)
    l1, g1 = gp.log_marginal_likelihood(theta, eval_gradient=True)
    l0, g0 = sk.log_marginal_likelihood(theta, eval_gradient=True)
    assert l1 == pytest.approx(l0, rel=1e-8)
    assert_allclose(g1, g0, rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("order", ["kernel_first", "white_first"])
def test_white_kernel_term_vs_sklearn(bo, order):
    """Sum(k, WhiteKernel): noise on the diagonal of K(X,X) and in the prior variance, nothing in K(X*,X)
    (SK/gaussian_process/kernels.py:1205-1330); LML, its gradient incl. d/dlog(noise), a full fit with restarts,
    predict(return_std / return_cov) against sklearn."""
    from sklearn.gaussian_process import GaussianProcessRegressor
    from sklearn.gaussian_process.kernels import ConstantKernel, WhiteKernel

    X, y = _synth(150, 3, 6)
    base = ConstantKernel(1.5) * Matern(nu=2.5, length_scale=0.8)
    k = base + WhiteKernel(0.05) if order == "kernel_first" else WhiteKernel(0.05) + base
    xt = np.random.RandomState(1).uniform(size=(40, 3))
    gp = bo.B200GaussianProcessRegressor(kernel=k, alpha=1e-8, normalize_y=True, optimizer=None).fit(X, y)
    sk = GaussianProcessRegressor(kernel=k, alpha=1e-8, normalize_y=True, optimizer=None).fit(X, y)
    mu, sd = gp.predict(xt, return_std=True)
    mu0, sd0 = sk.predict(xt, return_std=True)
    assert_allclose(mu, mu0, rtol=1e-7, atol=1e-9)
    assert_allclose(sd, sd0, rtol=1e-7, atol=1e-9)
    assert_allclose(gp.predict(xt[:9], return_cov=True)[1], sk.predict(xt[:9], return_cov=True)[1], rtol=1e-6, atol=1e-9)
    theta = k.theta + np.array([0.3, -0.2, 0.4][: k.theta.size])
    l1, g1 = gp.log_marginal_likelihood(theta, eval_gradient=True)
    l0, g0 = sk.log_marginal_likelihood(theta, eval_gradient=True)
    assert l1 == pytest.approx(l0, rel=1e-9)
    assert_allclose(g1, g0, rtol=1e-6, atol=1e-7)
    # full fit: same RandomState consumption and optimum to optimiser tolerance
    r1, r0 = np.random.RandomState(4), np.random.RandomState(4)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        gpf = bo.B200GaussianProcessRegressor(kernel=k, alpha=1e-8, normalize_y=True, n_restarts_optimizer=2,
                                              random_state=r1).fit(X, y)
        skf = GaussianProcessRegressor(kernel=k, alpha=1e-8, normalize_y=True, n_restarts_optimizer=2,
                                       random_state=r0).fit(X, y)
    assert r1.uniform() == r0.uniform()
    assert gpf.log_marginal_likelihood_value_ == pytest.approx(skf.log_marginal_likelihood_value_, rel=1e-6, abs=1e-6)
    assert_allclose(gpf.kernel_.theta, skf.kernel_.theta, rtol=0, atol=5e-3)


def test_bench_dump_outputs_are_the_last_timed_step(tmp_path):
    """bench.py --dump-outputs: with one timed step (warm-up >= 3 rotates back to candidate buffer 0) the dumped device
    records are the step whose result the JSON line reports; every file is float64."""
    import json
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "1", "--warmup", "3",
                          "--no-extra", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    j = json.loads(out.stdout.strip().splitlines()[-1])
    assert j["steps"] == 1
    d = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert sorted(d) == sorted(f"{leg}_{name}" for leg in ("device", "e2e")
                               for name in ("argmin_index", "argmin_value", "top_indices"))
    assert all(a.dtype == np.float64 for a in d.values())
    r = j["result"]
    assert int(d["device_argmin_index"]) == r["argmin_index"]
    assert_allclose(float(d["device_argmin_value"]), r["argmin_value"], rtol=1e-12, atol=0)
    assert [int(t) for t in d["device_top_indices"]] == r["top_indices"]
    assert d["e2e_top_indices"].shape == (10,)
