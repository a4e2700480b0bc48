"""How accurately can the gradient of the triangulated-point error be known at all?

The error is a small angle computed as th = sqrt(2 - 2 cos) (triangulation.cc:762-802), so the rounding of
cos (1e-16) is amplified by ~1/th^2 in d th. tests/test_callback_gpu.py compares the triangulated rows of J with
the compiled reference at 1e-6 instead of the 1e-9 used everywhere else; this file measures why:

  CPU   the reference's own _mrcal_triangulated_error() (oracle/_ref; its values are stored under tests/golden/)
        against a 60-digit evaluation (mpmath) of the same function: the reference's double-precision gradient
        is itself only good to ~1e-8..1e-7 relative at sub-milliradian angles, far from 1e-9
  GPU   our device function against the same 60-digit values: at least as close to the truth as the reference is

So a 1e-9 comparison between the two double-precision implementations would be comparing rounding noise."""
import ctypes as C

import numpy as np
import pytest

import problems

mp = pytest.importorskip("mpmath")


def _cases(n=40, seed=0):
    """Convergent ray pairs (no cheirality penalty), residual angles from ~1e-5 to ~1e-2 rad."""
    rng = np.random.default_rng(seed)
    out = []
    while len(out) < n:
        p = np.array((rng.uniform(-1, 1), rng.uniform(-1, 1), rng.uniform(3, 8)))      # the point, camera-0 coordinates
        t01 = np.array((rng.uniform(0.3, 1.5), rng.uniform(-0.2, 0.2), rng.uniform(-0.2, 0.2)))
        v0 = p * rng.uniform(0.5, 2.)
        v1 = (p - t01) * rng.uniform(0.5, 2.)
        # perturb one ray so that the two miss each other by a small angle
        v1 = v1 + np.linalg.norm(v1) * 10. ** rng.uniform(-5, -2) * rng.normal(size=3)
        out.append(np.concatenate((v0, v1, t01)))
    return np.array(out)


def _err_mp(v0, v1, t01):
    """_mrcal_triangulated_error() (triangulation.cc:958-1123), convergent branch, in mpmath."""
    cross = lambda a, b: (a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0])
    n2 = lambda a: a[0] * a[0] + a[1] * a[1] + a[2] * a[2]
    dot = lambda a, b: a[0] * b[0] + a[1] * b[1] + a[2] * b[2]
    p_recip = 1 / n2(cross(v0, v1))
    l0 = mp.sqrt(n2(cross(v1, t01)) * p_recip)
    l1 = mp.sqrt(n2(cross(v0, t01)) * p_recip)
    m = [(v0[i] * l0 + t01[i] + v1[i] * l1) / 2 for i in range(3)]
    costh = dot(v0, m) / mp.sqrt(n2(v0) * n2(m))
    return 2 * mp.sqrt(2 - 2 * abs(costh))


def _truth(case):
    mp.mp.dps = 60
    v0 = [mp.mpf(float(x)) for x in case[0:3]]
    v1 = [mp.mpf(float(x)) for x in case[3:6]]
    t = [mp.mpf(float(x)) for x in case[6:9]]
    err = _err_mp(v0, v1, t)
    g = []
    for k in range(6):
        def f(x, k=k):
            a, b = list(v1), list(t)
            if k < 3: a[k] = x
            else:     b[k - 3] = x
            return _err_mp(v0, a, b)
        g.append(mp.diff(f, v1[k] if k < 3 else t[k - 3]))
    return float(err), np.array([float(x) for x in g])


@pytest.fixture(scope="module")
def truth():
    cases = _cases()
    return cases, [_truth(c) for c in cases]


def _rel(g, g_true):
    return np.abs(g - g_true).max() / np.abs(g_true).max()


EPS = 2.2e-16


def _bound(err_true):
    # th = err/2 comes from th^2 = 2 - 2 cos: an absolute rounding error of a few eps in cos is a relative
    # error of a few eps / th^2 in th^2, in th and in its gradient
    th = err_true / 2.
    return 200. * EPS / (th * th) + 1e-12


def test_reference_gradient_precision(truth):
    cases, tr = truth
    gold = problems.oracle_golden("precision")
    assert np.array_equal(gold["cases"], cases)
    worst_grad = 0.
    for (e_true, g_true), e_g in zip(tr, gold["error_gradient"]):
        e = e_g[0]
        eg = _rel(e_g[1:], g_true)
        assert abs(e - e_true) / e_true <= _bound(e_true)
        assert eg <= _bound(e_true)
        if e_true > 1e-4:           # the residual angles a solve actually sees (0.3 px at f = 1500 is 2e-4 rad)
            worst_grad = max(worst_grad, eg)
    # THE FINDING: at realistic angles the reference's own double-precision gradient is off the exact one by
    # more than the 1e-9 gate used for the other rows -- and by less than the 1e-6 gate used for these
    assert 1e-9 < worst_grad < 1e-6, worst_grad


@pytest.mark.gpu
def test_device_gradient_precision(truth):
    from mrcal_b200 import _capi
    cases, tr = truth
    f = _capi.lib.mrcal_b200_debug_triangulated_error
    f.restype = C.c_bool
    out = np.zeros((len(cases), 7))
    inp = np.ascontiguousarray(cases)
    assert f(inp.ctypes.data_as(C.c_void_p), len(cases), out.ctypes.data_as(C.c_void_p)), _capi.last_error()
    for k, (c, (e_true, g_true)) in enumerate(zip(cases, tr)):
        # our device function is as close to the exact value and gradient as double precision allows -- the same
        # bound the reference meets
        assert abs(out[k, 0] - e_true) / e_true <= _bound(e_true)
        assert _rel(out[k, 1:], g_true) <= _bound(e_true)
