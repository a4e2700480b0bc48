"""CPU: the oracle for drt_cross_reprojection__dbpacked -- the reference's uncertainty.c compiled into oracle/_ref, on the
restated dpptrf_/dpptrs_ of oracle/stubs/ref_stubs.c -- against the DEFINITION it implements, written out densely in numpy
(uncertainty.c:21-127):  K = -pinv(Jcross) J_packed[frames, calobject_warp],  jcross_i = j_i[frame] Dinv M_frame,
M = d compose_rt(tiny, rt_ref_frame)/d tiny = [dr/dr0 0; -skew(t) I].
What the oracle returned (K, the packed state and, of the board rows of J in the frame and calobject_warp columns, the
Gram matrix: the definition needs no more of J) is stored under tests/golden/ by tests/golden/make_oracle_golden.py."""
import numpy as np
import pytest

import problems
from mrcal_b200 import synthetic

LENSMODELS = ["LENSMODEL_OPENCV4", "LENSMODEL_PINHOLE"]

SR, ST = 15. * np.pi / 180., 1.      # SCALE_ROTATION_FRAME, SCALE_TRANSLATION_FRAME (scales.h)


def _skew(t):
    return np.array([[0., -t[2], t[1]], [t[2], 0., -t[0]], [-t[1], t[0], 0.]])


def _dr_dr0(r):
    """mrcal_compose_r_tinyr0_gradientr0 (poseutils.c:1003-1062)"""
    B = np.linalg.norm(r) / 2.
    BtB = B / np.tan(B)
    return -np.outer(r, r) * (BtB - 1.) / (4. * B * B) + BtB * np.eye(3) - _skew(r) / 2.


def problem(lensmodel):
    kw, _ = synthetic.make_problem(lensmodel=lensmodel, Ncameras=3, Nframes=6, W=5, H=4, seed=2, pixel_noise=0.2)
    return kw


@pytest.mark.parametrize("lensmodel", LENSMODELS)
def test_rrp_against_the_definition(lensmodel):
    gold = problems.oracle_golden("cross_reprojection")
    K, b = gold[f"definition/{lensmodel}/K"], gold[f"definition/{lensmodel}/b"]
    i_f0, i_cw, Nmeas_obs, Nframes = gold[f"definition/{lensmodel}/layout"]
    cols = np.r_[i_f0:i_f0 + 6 * Nframes, i_cw:i_cw + 2]
    G = gold[f"definition/{lensmodel}/J_cols_gram"]          # Jobs_cols' Jobs_cols, Jobs_cols = J[:Nmeas_obs, cols]
    assert G.shape == (len(cols), len(cols)) and len(b) == K.shape[1]
    Dinv = np.diag([1. / SR] * 3 + [1. / ST] * 3)
    # Jcross = Jobs_cols T: each row sees one frame, the others add zeros
    T = np.zeros((len(cols), 6))
    for f in range(Nframes):
        q = b[i_f0 + 6 * f: i_f0 + 6 * f + 6]
        r, t = q[:3] * SR, q[3:] * ST
        M = np.block([[_dr_dr0(r), np.zeros((3, 3))], [-_skew(t), np.eye(3)]])
        T[6 * f: 6 * f + 6] = Dinv @ M
    # Jcross' Jcross = T' G T and Jcross' Jobs_cols = T' G
    K_np = -np.linalg.solve(T.T @ G @ T, T.T @ G)
    assert np.abs(K[:, cols] - K_np).max() <= 1e-9 * (1. + np.abs(K_np).max())
    rest = np.setdiff1d(np.arange(K.shape[1]), cols)
    assert not K[:, rest].any()
