"""mrcal_b200.cameramodel: the `.cameramodel` format either side of the solve (reference: mrcal/cameramodel.py,
native format). Host-only; runs without a GPU."""
import ast
import glob
import io
import os

import numpy as np
import pytest

import importlib

import mrcal_b200
import problems

# mrcal_b200.cameramodel is the CLASS (as mrcal.cameramodel is); the module holds the helpers too
cm = importlib.import_module("mrcal_b200.cameramodel")

# the reference's own model files (its test/data), stored as data fixtures
MODELS = os.path.join(problems.GOLDEN, "cameramodels")


def test_roundtrip_explicit_model():
    intr = np.array((1761.181055, 1761.250444, 1965.706996, 1087.518797, -0.0126, 0.0359, -0.00025, 0.00053, 0.0197, 0.0148,
                     -0.0562, 0.0500))
    m = cm.cameramodel(intrinsics=("LENSMODEL_OPENCV8", intr), imagersize=(4000, 2200),
                       rt_cam_ref=(2e-2, -3e-1, -1e-2, 1., 2., -3.), valid_intrinsics_region=((0, 0), (100, 0), (100, 50), (0, 0)))
    s = io.StringIO()
    m.write(s, note="written by a test\nsecond line")
    text = s.getvalue()
    assert text.startswith("# written by a test\n# second line\n{")
    m2 = cm.cameramodel(text)
    assert m2.intrinsics()[0] == "LENSMODEL_OPENCV8"
    assert np.allclose(m2.intrinsics()[1], intr, rtol=1e-9, atol=0)
    assert np.array_equal(m2.imagersize(), (4000, 2200)) and m2.imagersize().dtype == np.int32
    assert np.allclose(m2.rt_cam_ref(), (2e-2, -3e-1, -1e-2, 1., 2., -3.))
    assert np.allclose(m2.valid_intrinsics_region(), ((0, 0), (100, 0), (100, 50), (0, 0)))
    assert m2.optimization_inputs() is None and m2.icam_intrinsics() is None
    # both pose keys are written (mrcal < 2.5 reads 'extrinsics')
    d = ast.literal_eval(text)
    assert d["extrinsics"] == d["rt_cam_ref"] and list(d)[:2] == ["lensmodel", "intrinsics"]
    # the pose and its inverse
    rt = m2.rt_ref_cam()
    m2.rt_ref_cam(rt)
    assert np.allclose(m2.rt_cam_ref(), m.rt_cam_ref(), atol=1e-12)
    with pytest.raises(RuntimeError, match="needs 12 values"):
        cm.cameramodel(intrinsics=("LENSMODEL_OPENCV8", intr[:8]), imagersize=(10, 10))


def inverse_pose_inputs():
    return np.random.default_rng(0).normal(size=(5, 6))


def test_inverse_pose_matches_reference():
    gold = problems.oracle_golden("cameramodel")
    assert np.array_equal(gold["rt"], inverse_pose_inputs())
    for rt, inverted_ref in zip(gold["rt"], gold["inverted"]):
        assert np.allclose(cm.invert_rt(rt), inverted_ref, atol=1e-12)
    assert np.allclose(cm.invert_rt(np.array((0., 0., 0., 1., 2., 3.))), (0., 0., 0., -1., -2., -3.))


def test_model_from_a_solve_roundtrips_its_inputs(tmp_path):
    kw = dict(problems.golden_cases())["opencv8_points_fixed"]   # 3 cameras, camera 0 at the reference
    m = cm.cameramodel(optimization_inputs=kw, icam_intrinsics=2)
    assert m.icam_intrinsics() == 2 and m.icam_extrinsics() == 1
    assert np.array_equal(m.intrinsics()[1], kw["intrinsics"][2]) and np.array_equal(m.rt_cam_ref(), kw["rt_cam_ref"][1])
    assert cm.cameramodel(optimization_inputs=kw, icam_intrinsics=0).icam_extrinsics() == -1
    path = str(tmp_path / "cam2.cameramodel")
    m.write(path)
    m2 = cm.cameramodel(path)
    got = m2.optimization_inputs()
    for k, v in kw.items():
        if k == "do_apply_regularization_unity_cam01" and not v:
            assert k not in got   # new arguments at their default are not stored: older mrcal can then read the file
            continue
        if isinstance(v, np.ndarray):
            assert np.array_equal(got[k], v) and got[k].dtype == v.dtype, k
        else:
            assert got[k] == v, k
    # the pose arrays come back under both their names (files are written with the old ones)
    raw = np.load(io.BytesIO(__import__("base64").b85decode(m2._optimization_inputs_string)))
    assert "extrinsics_rt_fromref" in raw and "rt_cam_ref" not in raw
    assert got["frames_rt_toref"].startswith("ERROR:") and np.array_equal(got["rt_cam_ref"], kw["rt_cam_ref"])
    # None survives, and what was read can be solved again as it is
    d = dict(kw, calobject_warp=None)
    assert cm.deserialize_optimization_inputs(cm.serialize_optimization_inputs(d))["calobject_warp"] is None
    assert mrcal_b200.num_states(**got) == mrcal_b200.num_states(**kw)
    with pytest.raises(RuntimeError, match="icam_intrinsics is required"):
        cm.cameramodel(optimization_inputs=kw)


def test_legacy_names_and_errors():
    text = """{ 'distortion_model': 'DISTORTION_OPENCV4', 'intrinsics': [ 1000., 1000., 500., 400., 0.1, 0.2, 0.0, 0.0 ],
                'extrinsics': [ 0.1, 0.2, 0.3, 1, 2, 3 ], 'imagersize': [ 1000, 800 ] }"""
    m = cm.cameramodel(text)
    assert m.intrinsics()[0] == "LENSMODEL_OPENCV4" and np.allclose(m.rt_cam_ref(), (0.1, 0.2, 0.3, 1, 2, 3))
    with pytest.raises(cm.CameramodelParseException, match="NOT the same"):
        cm.cameramodel(text.replace("'imagersize'", "'rt_cam_ref': [ 0., 0., 0., 0., 0., 0. ], 'imagersize'"))
    with pytest.raises(cm.CameramodelParseException, match="missing"):
        cm.cameramodel("{ 'lensmodel': 'LENSMODEL_PINHOLE', 'intrinsics': [1., 1., 0., 0.] }")
    with pytest.raises(cm.CameramodelParseException, match="Failed to parse"):
        cm.cameramodel("{ this is not a model")
    with pytest.raises(cm.CameramodelParseException, match="icam_intrinsics or icam_extrinsics ARE given"):
        cm.cameramodel(text.replace("'imagersize'", "'icam_intrinsics': 0, 'imagersize'"))


def test_reads_the_reference_files():
    files = sorted(glob.glob(os.path.join(MODELS, "*.cameramodel")))
    assert files
    for path in files:
        m = cm.cameramodel(path)
        d = ast.literal_eval(open(path).read())
        lensmodel, intr = m.intrinsics()
        assert lensmodel == d.get("lensmodel", d.get("lens_model", d.get("distortion_model")))
        assert np.array_equal(intr, np.array(d["intrinsics"], float))
        assert len(intr) == mrcal_b200.lensmodel_num_params(lensmodel)
        assert np.array_equal(m.rt_cam_ref(), np.array(d.get("rt_cam_ref", d.get("extrinsics")), float))
        assert np.array_equal(m.imagersize(), d["imagersize"])
        # what this writes, this reads back the same
        again = cm.cameramodel(str(m))
        assert np.allclose(again.intrinsics()[1], intr, rtol=1e-9, atol=0)
