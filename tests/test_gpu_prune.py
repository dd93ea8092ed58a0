"""Pruned fused selection (DESIGN.md 4.1): candidates are screened on a partial variance bound and only those that
can still reach the top-k go through the full L^-1 K*^T product.  The records must equal, bit for bit, np.argmin /
stable argsort of the values the same engine returns when asked for them (that call never prunes), and the
executed-work counters must show that pruning happened."""
import ctypes as C
import types

import numpy as np
import pytest
from sklearn.gaussian_process.kernels import Matern

pytestmark = pytest.mark.gpu

CHUNK = 8 * 128 * 148  # rows per streamed chunk on a 148-SM B200


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


def _gp(bo, X, y, ls=0.7, alpha=1e-6, normalize_y=True):
    return bo.B200GaussianProcessRegressor(kernel=Matern(nu=2.5, length_scale=ls), alpha=alpha,
                                           normalize_y=normalize_y, optimizer=None).fit(X, y)


def _np_select(ys, k):
    return int(np.argmin(ys)), np.argsort(ys, kind="stable")[:k]


def _stats(bo):
    s, e = C.c_int64(), C.c_int64()
    bo._lib.check(bo._lib.lib().b200bo_last_select_stats(C.byref(s), C.byref(e)))
    return s.value, e.value


def _check_records(f, xt, k, ys=None):
    ys = f(xt) if ys is None else ys
    idx, val, top = f.argmin_topk(xt, k)
    ri, rtop = _np_select(ys, k)
    assert idx == ri
    assert val == ys[ri] or (np.isnan(val) and np.isnan(ys[ri]))
    assert list(top) == list(rtop)
    return ys


@pytest.fixture(scope="module")
def mid(bo):
    """N = 1024 (8 row blocks of L^-1), d = 4: the smallest model the pruned path takes."""
    X, y = _synth(1000, 4, 7)
    return X, y, _gp(bo, X, y, ls=0.5)


def test_c3_ei_records_exact_and_pruned(bo, monkeypatch):
    """bench.py's C3 problem at full size (d=16, N=4096, EI, 2^20 candidates of buffer 0), streamed and in one
    launch."""
    rs = np.random.RandomState(0)
    X = rs.uniform(size=(4096, 16))
    y = np.sin(X.sum(1)) + 0.1 * rs.randn(4096)
    f = bo.FusedAcquisition(bo._lib.ACQ_EI, _gp(bo, X, y), xi=0.01, y_max=float(y.max()))
    m = 1 << 20
    xt = np.random.RandomState(1000).uniform(size=(m, 16))
    ys = _check_records(f, xt, 10)
    screened, evaluated = _stats(bo)
    assert screened == m and evaluated < m // 10
    monkeypatch.setenv("B200BO_CHUNKED", "0")
    _check_records(f, xt, 10, ys)
    screened, evaluated = _stats(bo)
    assert screened == m and evaluated < m // 10


@pytest.mark.parametrize("k", [1, 10, 64])
def test_ei_k_and_exact_ties_of_the_kth_record(bo, mid, k):
    X, y, gp = mid
    f = bo.FusedAcquisition(bo._lib.ACQ_EI, gp, xi=0.01, y_max=float(y.max()))
    m = 1 << 17
    xt = np.random.RandomState(k).uniform(size=(m, 4))
    order = np.argsort(f(xt), kind="stable")
    kth = order[k - 1]
    for p in (3, m // 2 + 1, m - 1):  # copies of the k-th candidate in other tiles, before and after it
        if p != kth:
            xt[p] = xt[kth]
    ys = _check_records(f, xt, k)
    assert np.sum(ys == ys[kth]) >= 3
    screened, evaluated = _stats(bo)
    assert screened == m and evaluated < m // 2


@pytest.mark.parametrize("kind,kappa", [("ucb", 2.576), ("ucb", 0.0), ("poi", 0.0)])
def test_ucb_and_poi(bo, mid, kind, kappa):
    X, y, gp = mid
    m = 1 << 17
    xt = np.random.RandomState(11).uniform(size=(m, 4))
    if kind == "ucb":
        f = bo.FusedAcquisition(bo._lib.ACQ_UCB, gp, kappa=kappa)
    else:
        # y_max at the median mean: a = mu - y_max - xi is negative for half of the candidates, positive for the rest
        mu = gp.predict(xt[::64])
        f = bo.FusedAcquisition(bo._lib.ACQ_POI, gp, xi=0.0, y_max=float(np.median(mu)))
    _check_records(f, xt, 10)
    screened, evaluated = _stats(bo)
    assert screened == m and evaluated < m


def test_nan_values_survive(bo):
    """sigma clamped to 0 and a = 0 gives EI = NaN (0/0): np.argmin returns the FIRST NaN, argsort puts NaNs last;
    a NaN never has a usable bound, so it is always evaluated.  y_max = NaN makes every value NaN."""
    X, y = _synth(1000, 3, 3)
    gp = _gp(bo, X, y, ls=0.3, alpha=1e-12, normalize_y=False)
    m = 1 << 17
    xt = np.random.RandomState(0).uniform(size=(m, 3))
    xt[[90_000, 17, 129_000]] = X[[4, 9, 4]]
    mu = gp.predict(xt[[17]])
    f = bo.FusedAcquisition(bo._lib.ACQ_EI, gp, xi=0.0, y_max=float(mu[0]))
    ys = _check_records(f, xt, 8)
    assert _stats(bo)[0] == m
    f_nan = bo.FusedAcquisition(bo._lib.ACQ_EI, gp, xi=0.0, y_max=float("nan"))
    ys = _check_records(f_nan, xt, 8)
    assert np.isnan(ys).all()
    screened, evaluated = _stats(bo)
    assert screened == m and evaluated >= m


def test_philox_source(bo, O, mid):
    X, y, gp = mid
    f = bo.FusedAcquisition(bo._lib.ACQ_EI, gp, xi=0.01, y_max=float(y.max()))
    m, k, seed, base = 1 << 17, 10, 99, 5_000_000
    bounds = np.column_stack([np.zeros(4), np.ones(4)])
    bounds[1] = (-0.5, 1.5)
    idx, val, bx, top, tx = f.argmin_topk_philox(seed, bounds, m, k, index_base=base)
    screened, evaluated = _stats(bo)
    assert screened == m and evaluated < m // 2
    rows = O.philox_uniform(seed, base + np.arange(m), 4, bounds[:, 0], bounds[:, 1])
    ys = f(rows)
    ri, rtop = _np_select(ys, k)
    assert idx == base + ri and val == ys[ri] and list(top) == list(base + rtop)
    assert np.array_equal(bx, rows[ri]) and np.array_equal(tx, rows[rtop])


def test_streamed_host_batch(bo, mid, monkeypatch):
    """>= 2 chunks: every chunk is screened and compacted before its buffer is reused, the survivors of all
    chunks are evaluated once at the end.  Equal to the one-launch call and to numpy."""
    X, y, gp = mid
    f = bo.FusedAcquisition(bo._lib.ACQ_EI, gp, xi=0.01, y_max=float(y.max()))
    m = 2 * CHUNK + 12345
    xt = np.random.RandomState(5).uniform(size=(m, 4))
    xt[m - 3] = xt[100]
    a = f.argmin_topk(xt, 10)
    assert _stats(bo)[0] == m
    monkeypatch.setenv("B200BO_CHUNKED", "0")
    b = f.argmin_topk(xt, 10)
    assert _stats(bo)[0] == m
    assert a[0] == b[0] and a[1] == b[1] and list(a[2]) == list(b[2])
    ys = f(xt)
    ri, rtop = _np_select(ys, 10)
    assert a[0] == ri and list(a[2]) == list(rtop)


def test_ineligible_calls_take_the_full_launch(bo, mid):
    """Values requested alongside the records, or a constraint GP: no screen, every candidate evaluated."""
    from bayesianoptimization_b200 import _lib as B

    X, y, gp = mid
    m = 1 << 17
    xt = np.random.RandomState(2).uniform(size=(m, 4))
    f = bo.FusedAcquisition(B.ACQ_EI, gp, xi=0.01, y_max=float(y.max()))
    acq = np.empty(m)
    bv, bi = C.c_double(), C.c_int64()
    tv, ti = np.empty(10), np.empty(10, dtype=np.int64)
    B.check(B.lib().b200bo_acq_argmin_topk(C.byref(f.spec), B.as_dp(xt), m, 10, C.byref(bv), C.byref(bi),
                                           B.as_dp(tv), ti.ctypes.data_as(C.POINTER(C.c_int64)), B.as_dp(acq)))
    assert _stats(bo) == (0, m)
    ri, rtop = _np_select(acq, 10)
    assert bi.value == ri and list(ti) == list(rtop)
    cons = types.SimpleNamespace(model=[_gp(bo, X, np.cos(X.sum(1)), ls=0.5)], lb=[-0.5], ub=[0.5])
    fc = bo.FusedAcquisition(B.ACQ_EI, gp, constraint=cons, xi=0.01, y_max=float(y.max()))
    _check_records(fc, xt, 10)
    assert _stats(bo) == (0, m)
