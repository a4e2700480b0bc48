"""drt_cross_reprojection__dbpacked() on the GPU (mrcal_b200/csrc/cross_reprojection.cu) against the reference's own
_mrcal_drt_cross_reprojection__dbpacked() (uncertainty.c:798), compiled into oracle/_ref from the source where it lies
(LAPACK's dpptrf_/dpptrs_, restated in oracle/stubs/ref_stubs.c), fed the reference's own Jacobian; what it returned
is stored under tests/golden/ by tests/golden/make_oracle_golden.py. Gate: |K - K_ref| <= 1e-9 (1 + |K_ref|_max)."""
import numpy as np
import pytest

import mrcal_b200
import problems
from mrcal_b200 import synthetic

pytestmark = pytest.mark.gpu

SPL = "LENSMODEL_SPLINED_STEREOGRAPHIC_order=3_Nx=11_Ny=8_fov_x_deg=150"


def _clone(kw):
    return {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in kw.items()}


def _boards(lensmodel, Ncameras):
    kw, _ = synthetic.make_problem(lensmodel=lensmodel, Ncameras=Ncameras, Nframes=8, W=6, H=5, seed=4, pixel_noise=0.2)
    return kw, (-1, 0, 1, Ncameras - 1)


def _boards_with_outliers_and_locked_warp():
    kw, _ = synthetic.make_problem(lensmodel="LENSMODEL_OPENCV8", Ncameras=2, Nframes=6, W=5, H=4, seed=9, pixel_noise=0.3)
    flat = kw["observations_board"].reshape(-1, 3)
    flat[::17, 2] = -1.
    kw["do_optimize_calobject_warp"] = False
    return kw, (-1, 1)


def _points_only():
    kw, _ = synthetic.make_problem(lensmodel="LENSMODEL_OPENCV4", Ncameras=3, Nframes=2, W=6, H=5, seed=5, pixel_noise=0.2,
                                   Npoints=14, Npoints_fixed=3, which="all")
    for k in ("observations_board", "indices_frame_camintrinsics_camextrinsics", "rt_ref_frame", "calobject_warp"):
        kw.pop(k, None)
    kw["do_optimize_calobject_warp"] = False
    return kw, (-1, 0, 2)


def _config2_size():
    kw, _ = synthetic.baseline_config(2, pixel_noise=0.3)
    return kw, (-1, 1)


BOARDS = [("LENSMODEL_OPENCV4", 3), (SPL, 2), ("LENSMODEL_PINHOLE", 4)]


def cases():
    """{case: (optimization_inputs, icam_intrinsics values)}"""
    out = {f"boards_{lensmodel}_{Ncameras}": _boards(lensmodel, Ncameras) for lensmodel, Ncameras in BOARDS}
    out["boards_with_outliers_and_locked_warp"] = _boards_with_outliers_and_locked_warp()
    out["points_only"] = _points_only()
    out["config2_size"] = _config2_size()
    return out


def refused_problem():
    kw, _ = synthetic.make_problem(lensmodel="LENSMODEL_OPENCV4", Ncameras=3, Nframes=8, W=6, H=5, seed=4, pixel_noise=0.2,
                                   Npoints=12, Npoints_fixed=3, which="all")
    return kw


@pytest.fixture(scope="module")
def gold():
    return problems.oracle_golden("cross_reprojection")


def _check(gold, case, kw, icams):
    for icam in icams:
        K_ref = gold[f"{case}/{icam}"]
        K = mrcal_b200.drt_cross_reprojection__dbpacked(icam_intrinsics=icam, **_clone(kw))
        assert K.shape == K_ref.shape and K_ref.shape[0] == 6
        assert np.abs(K - K_ref).max() <= 1e-9 * (1. + np.abs(K_ref).max()), (icam, np.abs(K - K_ref).max())
        # the columns the reference leaves alone (intrinsics; in the rrp flavour the extrinsics; blocks the chosen camera
        # never sees) are exactly zero here too
        untouched = ~K_ref.any(axis=0)
        assert untouched.any() and not K[:, untouched].any()


@pytest.mark.parametrize("lensmodel,Ncameras", BOARDS)
def test_boards(gold, lensmodel, Ncameras):
    """rrp (icam_intrinsics = -1) and ccp for a camera at the reference (0: the frame path) and one with extrinsics"""
    _check(gold, f"boards_{lensmodel}_{Ncameras}", *_boards(lensmodel, Ncameras))


def test_boards_with_outliers_and_locked_warp(gold):
    _check(gold, "boards_with_outliers_and_locked_warp", *_boards_with_outliers_and_locked_warp())


def test_points_only(gold):
    """discrete points, no boards: the point path of rrp, and extrinsics x point of ccp"""
    _check(gold, "points_only", *_points_only())


def test_config2_size(gold):
    _check(gold, "config2_size", *_config2_size())


def test_refusals(gold):
    """what the reference refuses (uncertainty.c:944-989): boards and optimized points with a calobject_warp"""
    kw = refused_problem()
    assert gold["refused"]
    with pytest.raises(RuntimeError, match="calobject_warp"):
        mrcal_b200.drt_cross_reprojection__dbpacked(icam_intrinsics=-1, **_clone(kw))
