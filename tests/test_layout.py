"""State/measurement layout, lens-model descriptions and pack/unpack of the C-ABI
library versus what the compiled reference (oracle/_ref) computed, stored under tests/golden/.
Pure integer / scale logic: runs without a GPU. Model: the exact identities the
reference checks in test/test-basic-calibration.py:168-232."""
import ctypes as C
import itertools

import numpy as np
import pytest

import mrcal_b200
import problems
from mrcal_b200 import _capi

LENSMODELS = ("LENSMODEL_PINHOLE", "LENSMODEL_STEREOGRAPHIC", "LENSMODEL_LONLAT", "LENSMODEL_LATLON",
              "LENSMODEL_OPENCV4", "LENSMODEL_OPENCV5", "LENSMODEL_OPENCV8", "LENSMODEL_OPENCV12",
              "LENSMODEL_CAHVOR", "LENSMODEL_CAHVORE_linearity=0.37",
              problems.SPL3, problems.SPL2, problems.SPL3_BIG)


BAD_LENSMODELS = ("LENSMODEL_OPENCV7", "LENSMODEL_SPLINED_STEREOGRAPHIC", "LENSMODEL_SPLINED_STEREOGRAPHIC_order=3",
                  "LENSMODEL_SPLINED_STEREOGRAPHIC_order=3_Nx=30_Ny=20_fov_x_deg=170x", "LENSMODEL_CAHVORE", "",
                  "LENSMODEL_OPENCV8_")
SPLINED = (problems.SPL3, problems.SPL2, problems.SPL3_BIG)
PRECOMPUTED_LENSMODELS = SPLINED + ("LENSMODEL_OPENCV8",)
TRIANGULATED_CASES = ("tri_pinhole_only", "tri_opencv4_boards_points", "tri_stereographic_unity")


@pytest.fixture(scope="module")
def gold():
    return problems.oracle_golden("layout")


def test_lensmodel_parsing_matches_reference(gold):
    for i, name in enumerate(LENSMODELS):
        assert str(gold[f"lensmodel{i}/name"]) == name
        a = gold[f"lensmodel{i}/struct"].tobytes()
        b = mrcal_b200.api._lensmodel(name)
        assert a[:4] == bytes(b)[:4] and a[8:] == bytes(b)[8:], name
        assert int(gold[f"lensmodel{i}/num_params"]) == mrcal_b200.lensmodel_num_params(name)
        buf = C.create_string_buffer(256)
        assert _capi.lib.mrcal_lensmodel_name(buf, 256, C.byref(b))
        assert buf.value.decode() == str(gold[f"lensmodel{i}/written_name"])
    for i, bad in enumerate(BAD_LENSMODELS):
        ok_ref, type_ref, type_from_name_ref = gold[f"bad{i}"]
        rb = _capi.Lensmodel()
        ok = _capi.lib.mrcal_lensmodel_from_name(C.byref(rb), bad.encode())
        assert bool(ok_ref) == bool(ok) and type_ref == rb.type, bad
        with pytest.raises(RuntimeError):
            mrcal_b200.lensmodel_num_params(bad)
        assert type_from_name_ref == _capi.lib.mrcal_lensmodel_type_from_name(bad.encode())


def test_precomputed_lensmodel_data_matches_reference(gold):
    class Pre(C.Structure):
        _fields_ = [("ready", C.c_bool), ("segments_per_u", C.c_double)]
    for i, name in enumerate(PRECOMPUTED_LENSMODELS):
        ready_ref, segments_per_u_ref = gold[f"precomputed{i}"]
        b = Pre()
        _capi.lib._mrcal_precompute_lensmodel_data(C.byref(b), C.byref(mrcal_b200.api._lensmodel(name)))
        assert ready_ref and b.ready
        if "SPLINED" in name:
            assert segments_per_u_ref == b.segments_per_u and segments_per_u_ref > 0


def test_knots_match_reference(gold):
    for i, name in enumerate(SPLINED):
        ux, uy = mrcal_b200.knots_for_splined_models(name)
        assert np.array_equal(ux, gold[f"knots{i}/x"]) and np.array_equal(uy, gold[f"knots{i}/y"])


def _layout_numbers_product(kw):
    m = mrcal_b200
    out = [m.num_states(**kw), m.num_measurements(**kw), m.api._Inputs(dict(kw), for_layout_only=True).num_j_nonzero()]
    out += [m.num_states_intrinsics(**kw), m.num_states_extrinsics(**kw), m.num_states_frames(**kw),
            m.num_states_points(**kw), m.num_states_calobject_warp(**kw)]
    neg = lambda v: -1 if v is None else v
    out += [neg(m.state_index_intrinsics(0, **kw)), neg(m.state_index_intrinsics(1, **kw)),
            neg(m.state_index_extrinsics(0, **kw)), neg(m.state_index_extrinsics(1, **kw)),
            neg(m.state_index_frames(0, **kw)), neg(m.state_index_frames(2, **kw)),
            neg(m.state_index_points(0, **kw)), neg(m.state_index_points(3, **kw)),
            neg(m.state_index_calobject_warp(**kw))]
    out += [neg(m.measurement_index_boards(0, **kw)), neg(m.measurement_index_boards(2, **kw)),
            neg(m.measurement_index_points(0, **kw)), neg(m.measurement_index_points(1, **kw)),
            neg(m.measurement_index_regularization(**kw))]
    out += [m.num_measurements_boards(**kw), m.num_measurements_points(**kw), m.num_measurements_regularization(**kw)]
    return out


def test_layout_matches_stored_reference_numbers():
    g = np.load(problems.__file__.replace("problems.py", "golden/callback_cases.npz"))
    for name, kw in problems.golden_cases():
        assert _layout_numbers_product(kw) == list(g[f"{name}__layout"]), name


def layout_grid():
    """(what, optimization_inputs): all 2^7 selections x lens models x shapes, with zero-valued arrays."""
    rng = np.random.default_rng(0)
    shapes = [(1, 0, 3, 0, 0, 3, 0), (2, 1, 4, 0, 0, 6, 0), (3, 2, 2, 5, 2, 4, 9), (2, 2, 0, 4, 0, 0, 6), (4, 3, 5, 3, 3, 11, 5)]
    names = [n for n in _capi.SELECTION_BITS if n != "do_apply_outlier_rejection"]
    for lm in ("LENSMODEL_PINHOLE", "LENSMODEL_OPENCV8", "LENSMODEL_OPENCV12", "LENSMODEL_CAHVOR", problems.SPL3, problems.SPL2):
        Nintr = mrcal_b200.lensmodel_num_params(lm)
        for (Nci, Nce, Nf, Np, Npf, Nob, Nop) in shapes:
            idx_b = np.zeros((Nob, 3), np.int32)
            if Nob:
                idx_b[:, 0] = np.minimum(np.arange(Nob) * max(Nf, 1) // max(Nob, 1), max(Nf - 1, 0))
                idx_b[:, 1] = rng.integers(0, Nci, Nob)
                idx_b[:, 2] = rng.integers(-1, Nce, Nob)
            idx_p = np.zeros((Nop, 3), np.int32)
            if Nop:
                idx_p[:, 0] = rng.integers(0, max(Np, 1), Nop)
                idx_p[:, 1] = rng.integers(0, Nci, Nop)
                idx_p[:, 2] = rng.integers(-1, Nce, Nop)
            base = dict(lensmodel=lm, intrinsics=np.zeros((Nci, Nintr)), imagersizes=np.zeros((Nci, 2), np.int32),
                        rt_cam_ref=np.zeros((Nce, 6)), rt_ref_frame=np.zeros((Nf, 6)), points=np.zeros((Np, 3)),
                        observations_board=np.zeros((Nob, 3, 4, 3)), indices_frame_camintrinsics_camextrinsics=idx_b,
                        observations_point=np.zeros((Nop, 3)), indices_point_camintrinsics_camextrinsics=idx_p,
                        Npoints_fixed=Npf, calobject_warp=np.zeros(2), calibration_object_spacing=0.1)
            for bits in itertools.product((False, True), repeat=len(names)):
                yield (lm, Nci, Nce, Nf, Np, Npf, Nob, Nop, bits), dict(base, **dict(zip(names, bits)))


def test_layout_matches_compiled_reference_on_a_grid(gold):
    """All 2^7 selections x lens models x shapes, every layout function."""
    grid = gold["grid"]
    nchecked = 0
    for k, (what, kw) in enumerate(layout_grid()):
        assert _layout_numbers_product(kw) == list(grid[k]), what
        nchecked += 1
    assert nchecked == len(grid) and nchecked > 3000


def test_explicit_counts_interface():
    """Layout functions also take explicit counts instead of arrays (mrcal-pywrap.c:2164-2380);
    the identities of test/test-basic-calibration.py:168-232."""
    kw = dict(lensmodel="LENSMODEL_OPENCV4", Ncameras_intrinsics=4, Ncameras_extrinsics=3, Nframes=50,
              Nobservations_board=200, do_optimize_intrinsics_core=True, do_optimize_intrinsics_distortions=True,
              do_optimize_extrinsics=True, do_optimize_frames=True, do_optimize_calobject_warp=True)
    m = mrcal_b200
    assert m.state_index_intrinsics(2, **kw) == 8 * 2
    assert m.num_states_intrinsics(**kw) == 8 * 4
    assert m.num_intrinsics_optimization_params(**kw) == 8
    assert m.state_index_extrinsics(2, **kw) == 8 * 4 + 6 * 2
    assert m.num_states_extrinsics(**kw) == 6 * 3
    assert m.state_index_frames(35, **kw) == 8 * 4 + 6 * 3 + 6 * 35
    assert m.num_states_frames(**kw) == 6 * 50
    assert m.state_index_calobject_warp(**kw) == 8 * 4 + 6 * 3 + 6 * 50
    assert m.num_states_calobject_warp(**kw) == 2
    assert m.num_states(**kw) == 8 * 4 + 6 * 3 + 6 * 50 + 2
    assert m.state_index_points(0, **kw) is None
    assert m.state_index_frames(50, **kw) is None
    with pytest.raises(RuntimeError):
        m.num_states(Ncameras_intrinsics=1)   # lensmodel is required


def test_pack_unpack_matches_reference(gold):
    rng = np.random.default_rng(1)
    for name, kw in problems.golden_cases():
        # the reference's pack divides by the scale of each state and its unpack multiplies by it
        scale = gold[f"{name}/state_scale"]
        b = rng.normal(size=(3, len(scale)))
        mine = b.copy()
        mrcal_b200.pack_state(mine, **kw)
        theirs = b / scale
        assert np.array_equal(mine, theirs), name
        mrcal_b200.unpack_state(mine, **kw)
        theirs = theirs * scale
        assert np.array_equal(mine, theirs), name
        assert np.allclose(mine, b, rtol=1e-15, atol=0)
    with pytest.raises(RuntimeError):
        mrcal_b200.pack_state(np.zeros(3), **problems.golden_cases()[0][1])


def test_corresponding_icam_extrinsics():
    kw = dict(problems.golden_cases())["splined3_3cam_all"]   # 3 cameras, camera 0 at the reference
    assert mrcal_b200.corresponding_icam_extrinsics(0, **kw) == -1
    assert mrcal_b200.corresponding_icam_extrinsics(2, **kw) == 1


def test_triangulated_layout_and_validation(gold):
    """The layout functions with triangulated points need the SETS only (no rays, no GPU): compare with the
    compiled reference, and check the wrapper's complaints (mrcal-pywrap.c:1207-1240, 1406-1440)."""
    cases = dict(problems.golden_cases())
    for name in TRIANGULATED_CASES:
        kw = cases[name]
        num_measurements_ref, num_j_nonzero_ref = gold[f"{name}/num_measurements"]
        assert mrcal_b200.num_measurements(**kw) == num_measurements_ref
        assert mrcal_b200.api._Inputs(dict(kw), for_layout_only=True).num_j_nonzero() == num_j_nonzero_ref
        Ntri = mrcal_b200.num_measurements_points_triangulated(**kw)
        idx = kw["indices_point_triangulated_camintrinsics_camextrinsics"]
        assert Ntri == sum(n * (n - 1) // 2 for n in np.bincount(idx[:, 0]))
        m0 = mrcal_b200.measurement_index_points_triangulated(0, **kw)
        assert m0 == mrcal_b200.num_measurements_boards(**kw) + mrcal_b200.num_measurements_points(**kw)
        assert mrcal_b200.measurement_index_regularization(**kw) in (None, m0 + Ntri)
    kw = cases["tri_pinhole_only"]
    idx = kw["indices_point_triangulated_camintrinsics_camextrinsics"]

    def broken(f):
        bad = idx.copy()
        f(bad)
        return dict(kw, indices_point_triangulated_camintrinsics_camextrinsics=bad)

    # (the checks run where optimize()/optimizer_callback() parse their arguments; no GPU is touched before they pass)
    check = lambda k: mrcal_b200.api._Inputs(dict(k))
    check(kw)
    with pytest.raises(RuntimeError, match="consecutive and monotonic"):
        check(broken(lambda a: a.__setitem__((slice(None), 0), a[::-1, 0].copy())))
    with pytest.raises(RuntimeError, match="icam_intrinsics MUST be"):
        check(broken(lambda a: a.__setitem__((0, 1), 99)))
    with pytest.raises(RuntimeError, match="icam_extrinsics MUST be"):
        check(broken(lambda a: a.__setitem__((0, 2), 99)))
    lonely = np.concatenate((idx, np.array(((idx[-1, 0] + 1, 0, -1),), np.int32)))
    obs = np.concatenate((kw["observations_point_triangulated"], np.array(((1., 2., 1.),))))
    with pytest.raises(RuntimeError, match="at least 2 times"):
        check(dict(kw, indices_point_triangulated_camintrinsics_camextrinsics=lonely, observations_point_triangulated=obs))
    with pytest.raises(RuntimeError, match="Inconsistent Nobservations_point_triangulated"):
        check(dict(kw, observations_point_triangulated=obs))
