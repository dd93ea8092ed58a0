"""The reference's OWN driver on the device: two `bayes_opt.BayesianOptimization` objects are built from the
same seed, `bayesianoptimization_b200.enable()` is applied to one of them, and both are stepped through
suggest()/register() side by side (R/bayes_opt/bayesian_optimization.py:323-333, :262-281).  After every call:

  * the caller-owned RandomState is in the SAME state (the hooks consume the stream exactly like the
    reference: restarts of gp.fit, the candidate batch, GPHedge's softmax draw),
  * theta* of the hyper-parameter fit agrees to optimiser tolerance (two-tier parity, SURVEY.md section 7),
  * the B200 suggestion is the reference's suggestion to optimiser tolerance, and it is as good as the
    reference's under the REFERENCE's own acquisition closure (sklearn/scipy on the host).

Both optimizers then register the reference's point, so the trajectories stay comparable.  The vendored
package (oracle/_ref, oracle/vendor_ref.py) is the unmodified reference."""
import warnings

import numpy as np
import pytest
from numpy.testing import assert_allclose

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def bo():
    import bayesianoptimization_b200 as bo

    return bo


def readme_f(x, y):  # R/README.md:66-91
    return -(x**2) - (y - 1) ** 2 + 1


def _pair(ref, bo, seed, **kw):
    mk = lambda: ref.BayesianOptimization(random_state=seed, verbose=0, **kw)  # noqa: E731
    a, b = mk(), mk()
    bo.enable(b)
    return a, b


def _same_rng(a, b):
    sa, sb = a._random_state.get_state(), b._random_state.get_state()
    return sa[0] == sb[0] and np.array_equal(sa[1], sb[1]) and sa[2:] == sb[2:]


def _as_array(opt, params):
    return opt._space.params_to_array(params)


def _ref_closure_values(opt_ref, *points):
    """The reference's own (host) closure at the given points, after its suggest() fitted the GP."""
    acqf = opt_ref._acquisition_function
    base = getattr(acqf, "base_acquisition", acqf)
    f = base._get_acq(gp=opt_ref._gp, constraint=opt_ref._space.constraint)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return [float(f(p)[0]) for p in points]


def _step(a, b, f, constraint_f=None, tol=2e-3, check_rng=True, check_theta=True):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        sa = a.suggest()
        sb = b.suggest()
    xa, xb = _as_array(a, sa), _as_array(b, sb)
    if check_rng:
        assert _same_rng(a, b), "RandomState diverged: the device hooks consumed the stream differently"
    if check_theta:
        assert_allclose(b._gp.kernel_.theta, a._gp.kernel_.theta, rtol=0, atol=2e-3)
    span = a._space.bounds[:, 1] - a._space.bounds[:, 0]
    close = np.all(np.abs(xa - xb) <= tol * span)
    va, vb = _ref_closure_values(a, xa, xb)
    scale = max(abs(va), 1e-12)
    # same point to optimiser tolerance, or an equally good optimum under the reference's own closure
    assert close or vb <= va + 1e-4 * scale, (sa, sb, va, vb)
    kw = {}
    if constraint_f is not None:
        kw["constraint_value"] = constraint_f(**sa)
    for o in (a, b):
        o.register(params=sa, target=f(**sa), **kw)
    return sa, sb, close


def test_c1_readme_ucb_live(ref, bo):
    """BASELINE configs[0]: README 2-D function, default UCB(kappa=2.576), through the real driver."""
    a, b = _pair(ref, bo, 1, f=readme_f, pbounds={"x": (2, 4), "y": (-3, 3)})
    for o in (a, b):
        o.maximize(init_points=5, n_iter=0)
    assert _same_rng(a, b)
    n_close = 0
    for _ in range(6):
        sa, sb, close = _step(a, b, readme_f)
        n_close += close
    assert n_close >= 5
    assert isinstance(b._gp, bo.B200GaussianProcessRegressor) and isinstance(b._acquisition_function, bo.DeviceHooks)
    # BayesianOptimization.predict (bayesian_optimization.py:176-260) through the swapped GP
    pts = [{"x": 2.5, "y": 0.3}, {"x": 3.5, "y": -1.0}]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ma, sa_ = a.predict(pts, return_std=True, fit_gp=False)
        mb, sb_ = b.predict(pts, return_std=True, fit_gp=False)
    assert_allclose(mb, ma, rtol=1e-3, atol=1e-4)
    assert_allclose(sb_, sa_, rtol=1e-2, atol=1e-4)


def test_constrained_ei_live(ref, bo):
    """EI x constraint probability (R/bayes_opt/constraint.py:72-81, :153-221): target GP + constraint GP on
    the device, y_max over allowed points, same RNG stream (the constraint GPs re-seed from the int seed)."""
    from scipy.optimize import NonlinearConstraint

    def cf(x, y):
        return np.cos(x) * np.cos(y) - np.sin(x) * np.sin(y)

    def tf(x, y):
        return np.cos(2 * x) * np.cos(y) + np.sin(x)

    con = NonlinearConstraint(cf, -np.inf, 0.5)
    a, b = _pair(ref, bo, 3, f=tf, pbounds={"x": (0, 6), "y": (0, 6)}, constraint=con)
    for o in (a, b):
        o.maximize(init_points=6, n_iter=0)
    assert all(isinstance(m, bo.B200GaussianProcessRegressor) for m in b._space._constraint._model)
    for _ in range(5):
        _step(a, b, tf, constraint_f=cf, tol=5e-3)
    assert_allclose(b._space._constraint._model[0].kernel_.theta, a._space._constraint._model[0].kernel_.theta,
                    rtol=0, atol=1e-2)


def test_constant_liar_live(ref, bo):
    """ConstantLiar (R/bayes_opt/acquisition.py:1058-1148): several pending suggestions before any result."""
    A = ref.acquisition
    mk = lambda: A.ConstantLiar(A.UpperConfidenceBound(kappa=2.576), strategy="max")  # noqa: E731
    a = ref.BayesianOptimization(f=readme_f, pbounds={"x": (2, 4), "y": (-3, 3)}, acquisition_function=mk(),
                                 random_state=5, verbose=0)
    b = ref.BayesianOptimization(f=readme_f, pbounds={"x": (2, 4), "y": (-3, 3)}, acquisition_function=mk(),
                                 random_state=5, verbose=0)
    bo.enable(b)
    for o in (a, b):
        o.maximize(init_points=4, n_iter=0)
    for rnd in range(2):
        pend_a, pend_b = [], []
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            for _ in range(3):
                pend_a.append(a.suggest())
                pend_b.append(b.suggest())
        assert _same_rng(a, b)
        span = a._space.bounds[:, 1] - a._space.bounds[:, 0]
        for pa, pb in zip(pend_a, pend_b):
            assert np.all(np.abs(_as_array(a, pa) - _as_array(b, pb)) <= 5e-3 * span), (pa, pb)
        assert len(b._acquisition_function.dummies) == len(a._acquisition_function.dummies)
        # keep both on the reference's trajectory: same dummies, same registrations
        b._acquisition_function.dummies = [d.copy() for d in a._acquisition_function.dummies]
        for p in pend_a:
            for o in (a, b):
                o.register(params=p, target=readme_f(**p))


def test_gphedge_live(ref, bo):
    """GPHedge (R/bayes_opt/acquisition.py:1181-1360) through the driver with full hyper-parameter fits."""
    A = ref.acquisition
    mk = lambda: A.GPHedge([A.UpperConfidenceBound(kappa=2.0), A.ExpectedImprovement(xi=0.01),  # noqa: E731
                            A.ProbabilityOfImprovement(xi=0.01)])
    kw = dict(f=readme_f, pbounds={"x": (2, 4), "y": (-3, 3)}, verbose=0)
    a = ref.BayesianOptimization(acquisition_function=mk(), random_state=7, **kw)
    b = ref.BayesianOptimization(acquisition_function=mk(), random_state=7, **kw)
    bo.enable(b)
    for o in (a, b):
        o.maximize(init_points=5, n_iter=0)
    for _ in range(4):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            sa, sb = a.suggest(), b.suggest()
        assert _same_rng(a, b)
        ha, hb = a._acquisition_function, b._acquisition_function
        assert_allclose(hb.gains, ha.gains, rtol=1e-3, atol=1e-3)
        span = a._space.bounds[:, 1] - a._space.bounds[:, 0]
        assert np.all(np.abs(hb.previous_candidates - ha.previous_candidates) <= 5e-3 * span)
        assert np.all(np.abs(_as_array(a, sa) - _as_array(b, sb)) <= 5e-3 * span)
        hb.previous_candidates = ha.previous_candidates.copy()
        hb.gains = ha.gains.copy()
        for o in (a, b):
            o.register(params=sa, target=readme_f(**sa))


def test_int_and_categorical_parameters_live(ref, bo):
    """Mixed space: float + int (device np.round transform) + categorical (the reference's one-hot kernel
    transform applied on the host) through the DE + polish branch of _smart_minimize (:376-412)."""
    def f(x, k, c):
        return -((x - 2.0) ** 2) - 0.3 * (k - 3) ** 2 + {"a": 0.0, "b": 1.0, "c": -0.5}[c]

    pb = {"x": (0.0, 5.0), "k": (0, 6, int), "c": ["a", "b", "c"]}
    a, b = _pair(ref, bo, 11, f=f, pbounds=pb)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for o in (a, b):
            o.maximize(init_points=8, n_iter=0)
        for _ in range(3):
            sa, sb = a.suggest(), b.suggest()
            assert_allclose(b._gp.kernel_.theta, a._gp.kernel_.theta, rtol=0, atol=1e-2)
            xa, xb = _as_array(a, sa), _as_array(b, sb)
            va, vb = _ref_closure_values(a, xa, xb)
            same = sa["k"] == sb["k"] and sa["c"] == sb["c"] and abs(sa["x"] - sb["x"]) < 2e-2
            assert same or vb <= va + 1e-3 * max(abs(va), 1e-9), (sa, sb, va, vb)
            assert isinstance(sb["c"], str) and float(sb["k"]).is_integer()
            for o in (a, b):
                o.register(params=sa, target=f(**sa))
            b._random_state.set_state(a._random_state.get_state())  # DE consumes the stream per generation


def test_categorical_parameter_with_constraint_live(ref, bo):
    """Constraint GP + categorical parameter: target and constraint GPs both carry the space's one-hot kernel transform
    (two bound-method objects of the same TargetSpace, R/bayes_opt/target_space.py:105-111) and must share ONE transformed
    batch per device call.  (Found by the reference's own test_parameter.py on the drop-in; this pins it stepwise.)"""
    from scipy.optimize import NonlinearConstraint

    score = {"a": 0.0, "b": 1.0, "c": -0.5}

    def f(x, k, c):
        return -((x - 2.0) ** 2) - 0.3 * (k - 3) ** 2 + score[c]

    def g(x, k, c):
        return x + 0.5 * k - score[c]

    pb = {"x": (0.0, 5.0), "k": (0, 6, int), "c": ["a", "b", "c"]}
    a, b = _pair(ref, bo, 13, f=f, pbounds=pb, constraint=NonlinearConstraint(g, 0.5, 4.5))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for o in (a, b):
            o.maximize(init_points=8, n_iter=0)
        for _ in range(3):
            sa, sb = a.suggest(), b.suggest()
            xa, xb = _as_array(a, sa), _as_array(b, sb)
            va, vb = _ref_closure_values(a, xa, xb)
            same = sa["k"] == sb["k"] and sa["c"] == sb["c"] and abs(sa["x"] - sb["x"]) < 2e-2
            assert same or vb <= va + 1e-3 * max(abs(va), 1e-9), (sa, sb, va, vb)
            assert isinstance(sb["c"], str) and float(sb["k"]).is_integer()
            for o in (a, b):
                o.register(params=sa, target=f(**sa), constraint_value=g(**sa))
            b._random_state.set_state(a._random_state.get_state())  # DE consumes the stream per generation


def test_maximize_runs_end_to_end_on_device(ref, bo):
    """optimizer.maximize() (bayesian_optimization.py:348-391) on an enabled optimizer: runs, improves,
    every launch is the package's own."""
    from bayesianoptimization_b200 import _lib as B

    opt = ref.BayesianOptimization(f=readme_f, pbounds={"x": (2, 4), "y": (-3, 3)}, random_state=1, verbose=0)
    bo.enable(opt)
    n0 = B.lib().b200bo_launch_count()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        opt.maximize(init_points=3, n_iter=6)
    assert len(opt.space) == 9 and B.lib().b200bo_launch_count() > n0
    assert opt.max["target"] > -3.5  # the maximum on this domain is f(2, 1) = -3


def test_throughput_mode_candidate_source_through_the_driver(ref, bo):
    """enable(optimizer, candidate_source="device_philox"): the random candidates of suggest() are generated
    inside the fused kernel (no MT19937 stream, no H2D).  Opt-in: results are valid, not the reference's run."""
    from numpy.testing import assert_allclose

    opt = ref.BayesianOptimization(f=readme_f, pbounds={"x": (2, 4), "y": (-3, 3)}, random_state=1, verbose=0)
    bo.enable(opt, candidate_source="device_philox")
    a = opt._acquisition_function
    assert a.b200_candidate_source == "device_philox"
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        opt.maximize(init_points=4, n_iter=4)
        a._fit_gp(opt._gp, opt._space)
        f = a._get_acq(gp=opt._gp)
        x_min, v, seeds = a._random_sample_minimize(f, opt._space, np.random.RandomState(2), n_random=50_000, n_x_seeds=6)
    b = opt._space.bounds
    assert x_min.shape == (2,) and np.all(x_min >= b[:, 0]) and np.all(x_min <= b[:, 1])
    assert seeds.shape == (6, 2) and np.all(seeds >= b[:, 0]) and np.all(seeds <= b[:, 1])
    assert_allclose(f(x_min)[0], v, rtol=1e-9, atol=1e-12)          # the regenerated row is the evaluated row
    vals = f(seeds)
    assert np.all(np.diff(vals) >= -1e-12) and abs(vals[0] - v) <= 1e-9 * max(1.0, abs(v))
    assert opt.max["target"] > -3.5
