#!/usr/bin/env python
"""Side measurements for the rows next to the metric path (not the headline bench):
hyper-parameter fit (device LML + host L-BFGS-B) and a complete suggest() at BASELINE sizes."""
import json
import os
import sys
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle", "_ref"))  # the vendored, unmodified reference (oracle/vendor_ref.py)
import bayesianoptimization_b200 as bo  # noqa: E402
from bayes_opt.target_space import TargetSpace  # noqa: E402
from sklearn.gaussian_process.kernels import Matern  # noqa: E402

warnings.simplefilter("ignore")
out = {}
for n, d in [(1024, 8), (4096, 16)]:
    rs = np.random.RandomState(0)
    space = TargetSpace(None, {f"x{i:02d}": (0.0, 1.0) for i in range(d)})
    X = space.random_sample(n, rs)
    y = np.sin(X.sum(1)) + 0.1 * np.random.RandomState(0).randn(n)
    space._params, space._target = X, y
    gp = bo.B200GaussianProcessRegressor(kernel=Matern(nu=2.5), alpha=1e-6, normalize_y=True,
                                         n_restarts_optimizer=5, random_state=np.random.RandomState(1))
    L = bo._lib.lib()
    gp.fit(X[:256], y[:256])  # warm-up (allocations, module load)
    l0 = L.b200bo_launch_count()
    t0 = time.perf_counter()
    gp.fit(X, y)
    t_fit = time.perf_counter() - t0
    t0 = time.perf_counter()
    for _ in range(3):
        gp.log_marginal_likelihood(gp.kernel_.theta, eval_gradient=True)
    t_lml = (time.perf_counter() - t0) / 3
    acq = bo.ExpectedImprovement(xi=0.01)
    t0 = time.perf_counter()
    x = acq.suggest(gp, space, n_random=10_000, n_smart=10, fit_gp=False, random_state=np.random.RandomState(2))
    t_sug = time.perf_counter() - t0
    f = acq._get_acq(gp=gp)
    xt = space.random_sample(17, np.random.RandomState(3))
    f(xt)
    t0 = time.perf_counter()
    for _ in range(50):
        f(xt)
    t_stencil = (time.perf_counter() - t0) / 50
    t0 = time.perf_counter()
    for _ in range(50):
        f(xt[0])
    t_single = (time.perf_counter() - t0) / 50
    out[f"n{n}_d{d}"] = dict(fit_5restarts_s=t_fit, length_scale=float(gp.kernel_.length_scale),
                             lml_grad_eval_s=t_lml, suggest_nofit_s=t_sug,
                             acq_call_17pts_ms=1e3 * t_stencil, acq_call_1pt_ms=1e3 * t_single,
                             launches=int(L.b200bo_launch_count() - l0))
# the other BASELINE configs through the public call (host candidates in, argmin + 10 seeds out)
def _synth(n, d):
    r = np.random.RandomState(0)
    X = r.uniform(size=(n, d))
    return X, np.sin(X.sum(1)) + 0.1 * r.randn(n)


for tag, n, d, m, kind in [("c2_n1024_d8_ei", 1024, 8, 1 << 20, "ei"), ("c4_n2048_d16_poi_2constraints", 2048, 16, 1 << 19, "poi"),
                           ("c5_n8192_d32_ucb_shard", 8192, 32, 1 << 18, "ucb")]:
    X, y = _synth(n, d)
    gp = bo.B200GaussianProcessRegressor(kernel=Matern(nu=2.5, length_scale=0.7 if d < 32 else 1.0), alpha=1e-6,
                                         normalize_y=True, optimizer=None).fit(X, y)
    cm = None
    if kind == "poi":
        c = np.column_stack([np.cos(X.sum(1)), np.sin(2 * X.sum(1))])
        cm = bo.ConstraintModel(None, np.array([-np.inf, -0.5]), np.array([0.6, 0.5]))
        for mdl, l in zip(cm.model, (0.9, 0.5)):
            mdl.set_params(kernel=Matern(nu=2.5, length_scale=l), optimizer=None)
        cm.fit(X, c)
        a = bo.ProbabilityOfImprovement(xi=0.01)
        a.y_max = float(y[cm.allowed(c)].max())
    elif kind == "ei":
        a = bo.ExpectedImprovement(xi=0.01)
        a.y_max = float(y.max())
    else:
        a = bo.UpperConfidenceBound(kappa=2.576)
    f = a._get_acq(gp=gp, constraint=cm)
    xt = np.random.RandomState(1).uniform(size=(m, d))
    f.argmin_topk(xt[: m // 8], 10)
    t0 = time.perf_counter()
    f.argmin_topk(xt, 10)
    dt = time.perf_counter() - t0
    out[tag] = dict(candidates=m, seconds=dt, cand_per_s=m / dt, n_gps=1 if cm is None else 3)

# BASELINE configs[0]: README 2-D function, N=25, UCB - complete suggest() incl. the 6-start fit
def black_box(x, y):
    return -(x**2) - (y - 1) ** 2 + 1


space = TargetSpace(black_box, {"x": (2, 4), "y": (-3, 3)})
rs = np.random.RandomState(1)
for _ in range(25):
    space.probe(space.random_sample(random_state=rs))
gp = bo.B200GaussianProcessRegressor(kernel=Matern(nu=2.5), alpha=1e-6, normalize_y=True,
                                     n_restarts_optimizer=5, random_state=rs)
ucb = bo.UpperConfidenceBound(kappa=2.576)
ucb.suggest(gp, space, random_state=rs)
t0 = time.perf_counter()
for _ in range(3):
    ucb.suggest(gp, space, random_state=rs)
out["c1_readme_n25"] = dict(suggest_with_fit_s=(time.perf_counter() - t0) / 3)
try:
    from sklearn.gaussian_process import GaussianProcessRegressor as SkGPR

    skgp = SkGPR(kernel=Matern(nu=2.5), alpha=1e-6, normalize_y=True, n_restarts_optimizer=5, random_state=rs)
    t0 = time.perf_counter()
    skgp.fit(space.params, space.target)
    out["c1_readme_n25"]["sklearn_fit_only_s"] = time.perf_counter() - t0
except Exception:
    pass
print(json.dumps(out))
