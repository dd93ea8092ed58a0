"""pytest plugin: run the reference's OWN test modules against the drop-in.

    python -m pytest -p tests.ref_suite_plugin oracle/_ref/ref_tests

The reference's tests (vendored, unmodified, into the git-ignored oracle/_ref/ref_tests by oracle/vendor_ref.py)
build their objects from three names: ``sklearn.gaussian_process.GaussianProcessRegressor``, the classes of
``bayes_opt.acquisition`` and ``bayes_opt.constraint.ConstraintModel``.  Before those modules are collected this
plugin rebinds the names to the B200 classes (which ARE the reference's classes + the device hooks), so every
``acq.suggest(gp, target_space)``, ``BayesianOptimization.suggest()/maximize()``, ``ConstraintModel.predict`` of
the reference's suite runs on the device, and the reference's own assertions judge the result.  Nothing under
oracle/_ref is edited.  Used by tests/test_gpu_reference_suite.py (GPU) and, with B200BO_REF_SUITE_DRYRUN=1, by a
CPU test that only checks the rebinding itself.
"""
from __future__ import annotations

import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "oracle", "_ref"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

REBOUND = {}
DEVICE_CALLS = {}


def rebind():
    import sklearn.gaussian_process as skgp
    import bayes_opt
    from bayes_opt import acquisition as racq, bayesian_optimization as rbo, constraint as rcon, target_space as rts

    import bayesianoptimization_b200 as b200
    from bayesianoptimization_b200 import acquisition as bacq

    gp_cls = b200.B200GaussianProcessRegressor
    for mod in (skgp, rbo, rcon):
        if hasattr(mod, "GaussianProcessRegressor"):
            REBOUND[f"{mod.__name__}.GaussianProcessRegressor"] = mod.GaussianProcessRegressor
            mod.GaussianProcessRegressor = gp_cls
    for name in ("AcquisitionFunction", "UpperConfidenceBound", "ProbabilityOfImprovement", "ExpectedImprovement",
                 "ConstantLiar", "GPHedge"):
        REBOUND[f"bayes_opt.acquisition.{name}"] = getattr(racq, name)
        setattr(racq, name, getattr(bacq, name))
    for mod in (rcon, rbo, rts, bayes_opt):
        if hasattr(mod, "ConstraintModel"):
            REBOUND[f"{mod.__name__}.ConstraintModel"] = mod.ConstraintModel
            mod.ConstraintModel = b200.ConstraintModel
    # evidence for the log: how often the suite reached the device entry points
    from bayesianoptimization_b200.fused import FusedAcquisition
    for cls, names in ((gp_cls, ("fit", "predict", "log_marginal_likelihood")),
                       (FusedAcquisition, ("__call__", "argmin_topk"))):
        for name in names:
            _count(cls, name)
    return REBOUND


def _count(cls, name):
    inner = getattr(cls, name)
    key = f"{cls.__name__}.{name}"
    DEVICE_CALLS[key] = 0

    def counted(*a, **k):
        DEVICE_CALLS[key] += 1
        return inner(*a, **k)

    counted.__name__ = name
    counted.__doc__ = inner.__doc__
    setattr(cls, name, counted)


def pytest_configure(config):
    rebind()


def pytest_terminal_summary(terminalreporter):
    terminalreporter.write_line("b200 drop-in: rebound " + ", ".join(sorted(REBOUND)))
    terminalreporter.write_line("b200 drop-in: device entry points reached: "
                                + ", ".join(f"{k} x{v}" for k, v in sorted(DEVICE_CALLS.items())))
