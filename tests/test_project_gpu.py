"""mrcal_project() / mrcal_unproject() of the C-ABI library (mrcal_b200/csrc/project.cu) against the compiled
reference: values and dq/dp of every lens model, the closed-form unprojections directly, the iterative ones
through the reference's own project() (the reference's iterative unproject needs libdogleg, which the oracle
build stubs out: oracle/ref.py unproject()). What the reference returned is stored under tests/golden/ by
tests/golden/make_oracle_golden.py."""
import numpy as np
import pytest

import mrcal_b200
import problems
from mrcal_b200 import synthetic

pytestmark = pytest.mark.gpu

MODELS = ("LENSMODEL_PINHOLE", "LENSMODEL_STEREOGRAPHIC", "LENSMODEL_LONLAT", "LENSMODEL_LATLON",
          "LENSMODEL_OPENCV4", "LENSMODEL_OPENCV5", "LENSMODEL_OPENCV8", "LENSMODEL_OPENCV12", "LENSMODEL_CAHVOR",
          "LENSMODEL_CAHVORE_linearity=0.37", "LENSMODEL_CAHVORE_linearity=-0.25",
          "LENSMODEL_SPLINED_STEREOGRAPHIC_order=3_Nx=8_Ny=6_fov_x_deg=100",
          "LENSMODEL_SPLINED_STEREOGRAPHIC_order=2_Nx=8_Ny=6_fov_x_deg=100")


def intrinsics(lm, unproject):
    intr = synthetic.true_intrinsics(lm, 1, np.random.default_rng(0))[0]
    if unproject and lm.startswith("LENSMODEL_CAHVORE"):
        intr[-3:] = 0.   # the reference only unprojects central models (mrcal.c:3203-3214)
    return intr


@pytest.fixture(scope="module")
def gold():
    return problems.oracle_golden("project")


def _points(n, seed):
    rng = np.random.default_rng(seed)
    p = rng.uniform(-1., 1., (n, 3))
    p[:, 2] += 3.
    return p


@pytest.mark.parametrize("lm", MODELS)
def test_project_matches_reference(gold, lm):
    intr = intrinsics(lm, unproject=False)
    p = _points(40, 1)
    q_ref, g_ref = gold[f"{lm}/q"], gold[f"{lm}/dq_dp"]
    q, g, gi = mrcal_b200.project(p, lm, intr, get_gradients=True)
    assert np.abs(q - q_ref).max() <= 1e-9 * (1. + np.abs(q_ref).max())
    assert np.abs(g - g_ref).max() <= 1e-9 * (1. + np.abs(g_ref).max())
    # the gradient with respect to the intrinsics: dense (N,2,Nintrinsics), mrcal.c:2866-2992
    g3, gi_ref = gold[f"{lm}/dq_dp_with_intrinsics"], gold[f"{lm}/dq_dintrinsics"]
    assert gi.shape == gi_ref.shape == (40, 2, len(intr))
    assert np.abs(gi - gi_ref).max() <= 1e-9 * (1. + np.abs(gi_ref).max())
    assert np.abs(g - g3).max() <= 1e-9 * (1. + np.abs(g3).max())
    # broadcasting over leading dimensions, and the no-gradient flavour
    q2 = mrcal_b200.project(p.reshape(8, 5, 3), lm, intr)
    # (another instantiation of the kernel: the compiler contracts its multiply-adds differently, last-bit differences)
    assert q2.shape == (8, 5, 2) and np.abs(q2.reshape(-1, 2) - q).max() <= 1e-12 * (1. + np.abs(q).max())


@pytest.mark.parametrize("lm", MODELS)
def test_unproject(gold, lm):
    intr = intrinsics(lm, unproject=True)
    p = _points(40, 2)
    q = gold[f"{lm}/unproject_q"]       # the reference's projection of p
    v = mrcal_b200.unproject(q, lm, intr)
    v_ref = gold[f"{lm}/unproject_v"]
    n = lambda a: a / np.linalg.norm(a, axis=-1, keepdims=True)
    assert np.abs(n(v) - n(p)).max() < 1e-9           # it inverts the projection
    assert np.abs(v - v_ref).max() < 1e-9             # ... with the reference's scale convention
    # (projected by this library, whose projection test_project_matches_reference pins to the reference's at 1e-9)
    assert np.abs(mrcal_b200.project(v, lm, intr) - q).max() < 1e-8


def test_unproject_refuses_noncentral_cahvore():
    lm = "LENSMODEL_CAHVORE_linearity=0.37"
    intr = synthetic.true_intrinsics(lm, 1, np.random.default_rng(0))[0]
    with pytest.raises(RuntimeError, match="central"):
        mrcal_b200.unproject(np.array(((100., 200.),)), lm, intr)


def test_unproject_reports_failure_as_nan():
    # a pixel no ray projects to: with only k4 = 1 the radial map is r / (1 + r^2) <= 0.5, and this pixel sits
    # at 5. NaN x,y, as mrcal.c:3247-3262
    lm = "LENSMODEL_OPENCV8"
    intr = np.array((1000., 1000., 500., 500., 0., 0., 0., 0., 0., 1., 0., 0.))
    v = mrcal_b200.unproject(np.array(((5500., 500.), (600., 520.))), lm, intr)
    assert np.isnan(v[0, 0]) and np.isnan(v[0, 1])
    assert np.isfinite(v[1]).all()
