"""Parity of the CUDA cost function (residuals x + CSR Jacobian) with the
reference's optimizer_callback(), called through the reference-named C-ABI
entry point mrcal_optimizer_callback() (via mrcal_b200.optimizer_callback).

Gate (BASELINE.md / SURVEY.md 8d): |x-x_ref| <= 1e-9 (1+|x_ref|),
|J-J_ref| <= 1e-9 (1+|J_ref|) per entry, CSR structure (p, i) identical."""
import hashlib
import os

import numpy as np
import pytest

import mrcal_b200
import problems
from mrcal_b200 import synthetic
from test_oracle_golden import optimizer_callback_golden_case

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
TOL = 1e-9


def assert_close(a, b, what, tol=TOL):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    err = np.abs(a - b) / (1. + np.abs(b))
    assert err.size == 0 or err.max() <= tol, f"{what}: worst relative-to-scale error {err.max():.3g} at {err.argmax()}"


@pytest.mark.parametrize("name,kw", problems.golden_cases(), ids=[c[0] for c in problems.golden_cases()])
def test_callback_matches_stored_reference_output(name, kw):
    g = np.load(os.path.join(GOLDEN, "callback_cases.npz"))
    b, x, J, _ = mrcal_b200.optimizer_callback(**kw, no_factorization=True)
    assert J.indptr.dtype == np.int32 and J.indices.dtype == np.int32
    assert np.array_equal(J.indptr, g[f"{name}__Jp"]), "row pointers differ"
    assert np.array_equal(J.indices, g[f"{name}__Ji"]), "column indices differ"
    assert_close(b, g[f"{name}__b"], "b_packed")
    assert_close(x, g[f"{name}__x"], "x")
    if "observations_point_triangulated" in kw:
        # The triangulated error is a small angle th = sqrt(2 - 2 cos) (triangulation.cc:781-817): the rounding of
        # cos (1e-16) is amplified by 1/th^2 ~ 1e8 in d th, in the reference as much as here. The other rows
        # keep the 1e-9 gate; these gradients agree to the accuracy either implementation has
        m0 = mrcal_b200.measurement_index_points_triangulated(0, **kw)
        m1 = m0 + mrcal_b200.num_measurements_points_triangulated(**kw)
        j0, j1 = J.indptr[m0], J.indptr[m1]
        assert_close(J.data[:j0], g[f"{name}__Jx"][:j0], "J values before the triangulated rows")
        assert_close(J.data[j1:], g[f"{name}__Jx"][j1:], "J values after the triangulated rows")
        assert_close(J.data[j0:j1], g[f"{name}__Jx"][j0:j1], "J values of the triangulated rows", tol=1e-6)
    else:
        assert_close(J.data, g[f"{name}__Jx"], "J values")
    # no_jacobian path gives the same x
    b2, x2, J2, f2 = mrcal_b200.optimizer_callback(**kw, no_jacobian=True, no_factorization=True)
    assert J2 is None and f2 is None
    assert np.allclose(x, x2, rtol=1e-13, atol=1e-12) and np.array_equal(b, b2)


@pytest.mark.parametrize("i", range(6))
def test_callback_matches_reference_golden_vectors(i):
    """The reference's own regression vectors (test/test-optimizer-callback.py), rows below
    the regularization index (the stored regularization rows predate today's scales)."""
    kw, x_ref, J_ref = optimizer_callback_golden_case(i)
    b, x, J, _ = mrcal_b200.optimizer_callback(**kw, no_factorization=True)
    Jd = J.toarray()
    mrcal_b200.pack_state(Jd, **kw)
    ireg = mrcal_b200.measurement_index_regularization(**kw)
    n = ireg if ireg is not None else len(x)
    assert x.shape == x_ref.shape and Jd.shape == J_ref.shape
    assert_close(x[:n], x_ref[:n], "x")
    assert_close(Jd[:n], J_ref[:n], "J (unpacked)")
    # the reference test's own bar: RMS error <= 1e-6 (test/testutils.py:113-260)
    assert np.sqrt(np.mean((x[:n] - x_ref[:n]) ** 2)) < 1e-6
    assert np.sqrt(np.mean((Jd[:n] - J_ref[:n]) ** 2)) < 1e-6
    # unpack(pack(J)) == J (test-optimizer-callback.py:163-172)
    J2 = J.toarray()
    mrcal_b200.pack_state(J2, **kw)
    mrcal_b200.unpack_state(J2, **kw)
    assert np.allclose(J2, J.toarray(), rtol=1e-14, atol=0)


BASELINE_CONFIGS = [1, 2, 3, 5]


def structure_digest(indptr, indices):
    h = hashlib.sha256()
    for a in (indptr, indices):
        h.update(np.ascontiguousarray(a, np.int32).tobytes())
    return h.hexdigest()


def sample_indices(n, k=512):
    """A fixed sample of k entries of an output of length n: the first, the last and a seeded draw between."""
    if n <= k:
        return np.arange(n, dtype=np.int32)
    return np.unique(np.r_[0, n - 1, np.random.default_rng(n).choice(n, k - 2, replace=False)]).astype(np.int32)


@pytest.mark.parametrize("config", BASELINE_CONFIGS)
def test_callback_matches_compiled_reference_at_baseline_sizes(config):
    """BASELINE.json configs 1-3 and 5 at full size against the compiled reference (oracle/_ref). The CSR structure
    is compared whole (by digest); b, x and the values of J at a fixed sample of 512 entries each
    (tests/golden/make_oracle_golden.py)."""
    gold = problems.oracle_golden("callback")
    kw, _ = synthetic.baseline_config(config)
    b, x, J, _ = mrcal_b200.optimizer_callback(**kw, no_factorization=True)
    assert (len(b), len(x), J.nnz) == tuple(gold[f"config{config}/shape"])
    assert structure_digest(J.indptr, J.indices) == str(gold[f"config{config}/structure_sha256"])
    for what, v in (("b", b), ("x", x), ("Jx", J.data)):
        i = gold[f"config{config}/{what}_index"]
        assert np.array_equal(i, sample_indices(len(v)))
        assert_close(v[i], gold[f"config{config}/{what}"], {"b": "b_packed", "x": "x", "Jx": "J values"}[what])
    if config == 3:
        assert (len(b), len(x), J.nnz) == (7220, 324800, 9129600)   # SURVEY.md 8 table


def test_projection_known_answers():
    """The reference's in-source projection known answers (test/test-projections.py:337-514): project the given
    camera-frame points with the given intrinsics. Done through the real path: a one-camera problem whose fixed
    points sit at p, observed at pixel (0,0) with weight 1, so that x = q."""
    g = np.load(os.path.join(GOLDEN, "projections.npz"))
    ntested = 0
    for i in range(int(g["N"])):
        lm = str(g[f"lensmodel_{i}"])
        intr, p, q_ref = g[f"intrinsics_{i}"], g[f"p_{i}"], g[f"q_{i}"]
        for k in range(p.shape[0]):
            ii = np.ascontiguousarray((intr[k] if intr.ndim == 2 else intr)[None, :])
            kw = dict(lensmodel=lm, intrinsics=ii, imagersizes=np.array(((4000, 2200),), np.int32),
                      points=np.ascontiguousarray(p[k:k + 1]), Npoints_fixed=1,
                      observations_point=np.array(((0., 0., 1.),)),
                      indices_point_camintrinsics_camextrinsics=np.array(((0, 0, -1),), np.int32),
                      do_optimize_intrinsics_core=True, do_optimize_intrinsics_distortions=False,
                      do_optimize_frames=False, do_apply_regularization=False)
            x = mrcal_b200.optimizer_callback(**kw, no_jacobian=True, no_factorization=True)[1]
            assert np.abs(x[:2] - q_ref[k]).max() < 2e-6 * max(1., np.abs(q_ref[k]).max()), (lm, k, x[:2], q_ref[k])
            ntested += 1
    assert ntested >= 36


def test_callback_size_independent_properties():
    """Full-size config 3 without the oracle: perfect observations give zero board residuals
    (test-basic-calibration.py:371-382) and J predicts finite differences of x."""
    kw, truth = synthetic.baseline_config(3)
    kw_true = dict(kw, intrinsics=truth["intrinsics"], rt_cam_ref=truth["rt_cam_ref"],
                   rt_ref_frame=truth["rt_ref_frame"], calobject_warp=truth["calobject_warp"])
    x = mrcal_b200.optimizer_callback(**kw_true, no_jacobian=True, no_factorization=True)[1]
    nb = mrcal_b200.num_measurements_boards(**kw)
    assert np.abs(x[:nb]).max() < 1e-8
    P = mrcal_b200.Problem(**kw)
    b0, x0, J = P.callback()
    rng = np.random.default_rng(0)
    db = rng.normal(size=b0.shape) * 1e-6
    P.reset(b0 + db)
    x1 = P.callback(jacobian=False)[1]
    P.reset(b0 - db)
    x2 = P.callback(jacobian=False)[1]
    lin = J @ db
    assert np.abs((x1 - x2) / 2. - lin).max() < 1e-6 * np.abs(lin).max() + 1e-9
    # reset() with no argument returns to the seed
    P.reset()
    assert np.allclose(P.callback(jacobian=False)[1], x0, rtol=1e-13, atol=1e-12)


def test_callback_error_behaviour():
    kw, _ = synthetic.make_problem(Ncameras=2, Nframes=3, W=4, H=4)
    with pytest.raises(RuntimeError, match="Unknown keyword"):
        mrcal_b200.optimizer_callback(**kw, bogus=1)
    bad = dict(kw, intrinsics=kw["intrinsics"].astype(np.float32))
    with pytest.raises(RuntimeError, match="dtype"):
        mrcal_b200.optimizer_callback(**bad)
    bad = dict(kw, indices_frame_camintrinsics_camextrinsics=kw["indices_frame_camintrinsics_camextrinsics"][::-1].copy())
    with pytest.raises(RuntimeError, match="monotonically|sequentially"):
        mrcal_b200.optimizer_callback(**bad)
    bad = dict(kw, lensmodel="LENSMODEL_SPLINED_STEREOGRAPHIC_order=4_Nx=8_Ny=6_fov_x_deg=100", intrinsics=np.zeros((2, 4 + 2 * 48)))
    with pytest.raises(RuntimeError, match="no CUDA implementation"):
        mrcal_b200.optimizer_callback(**bad)
    # None-valued kwargs are ignored, as in the reference (mrcal-pywrap.c:1491-1555)
    mrcal_b200.optimizer_callback(**kw, points=None, imagepaths=None, no_factorization=True)
