"""Small seeded problems shared by the golden-fixture generator and the tests.

Every case is rebuilt from mrcal_b200.synthetic.make_problem() with a fixed seed,
so the inputs exist wherever the repo does; tests/golden/callback_cases.npz holds
what the COMPILED REFERENCE computed for them (tests/golden/make_golden.py)."""
import os

import numpy as np

from mrcal_b200 import synthetic

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

SPL3 = "LENSMODEL_SPLINED_STEREOGRAPHIC_order=3_Nx=11_Ny=8_fov_x_deg=150"
SPL2 = "LENSMODEL_SPLINED_STEREOGRAPHIC_order=2_Nx=12_Ny=9_fov_x_deg=150"
SPL3_BIG = "LENSMODEL_SPLINED_STEREOGRAPHIC_order=3_Nx=30_Ny=20_fov_x_deg=170"


def _sel(core, dist, extr, frames, warp, reg=True, unity=False):
    return dict(do_optimize_intrinsics_core=core, do_optimize_intrinsics_distortions=dist,
                do_optimize_extrinsics=extr, do_optimize_frames=frames, do_optimize_calobject_warp=warp,
                do_apply_regularization=reg, do_apply_regularization_unity_cam01=unity)


def _mark_outliers(inputs, n, seed):
    rng = np.random.default_rng(seed)
    o = inputs["observations_board"]
    flat = o.reshape(-1, 3)
    i = rng.choice(flat.shape[0], n, replace=False)
    flat[i, 2] *= -1.
    return inputs


def add_triangulated_points(inp, truth, Npoints, seed, pixel_noise=0.3, outliers=1):
    """Triangulated-point observations (the reference's SfM-style measurements, mrcal.c:5180-5653) for an
    existing problem: Npoints world points, each seen by 2 or more of the cameras; pixels = projection with
    the problem's (locked) intrinsics + noise; weight <= 0 marks an outlier."""
    rng = np.random.default_rng(seed)
    Ncam = inp["intrinsics"].shape[0]
    rt_all = np.concatenate((np.zeros((1, 6)), truth["rt_cam_ref"]))   # camera 0 sits at the reference
    # in front of the middle of the rig
    centre = np.mean([-synthetic.R_from_r(rt[:3]).T @ rt[3:] for rt in rt_all], axis=0)
    obs, idx = [], []
    for ipt in range(Npoints):
        p_ref = centre + np.array((rng.uniform(-1., 1.), rng.uniform(-0.7, 0.7), rng.uniform(4., 8.)))
        cams = np.sort(rng.choice(Ncam, size=rng.integers(2, Ncam + 1), replace=False))
        for icam in cams:
            p_cam = synthetic.transform_rt(rt_all[icam], p_ref)
            q = synthetic.project(p_cam, inp["lensmodel"], inp["intrinsics"][icam]) + rng.normal(0, pixel_noise, 2)
            obs.append((q[0], q[1], 1.0))
            idx.append((ipt, icam, icam - 1))
    obs = np.array(obs)
    if outliers:
        obs[rng.choice(obs.shape[0], outliers, replace=False), 2] = np.array((-1., 0.))[np.arange(outliers) % 2]
    inp["observations_point_triangulated"] = obs
    inp["indices_point_triangulated_camintrinsics_camextrinsics"] = np.array(idx, np.int32)
    return inp


def golden_cases():
    """(name, optimization_inputs). Small: the whole set evaluates in seconds."""
    cases = []

    def add(name, lensmodel, Ncameras, Nframes, sel=None, W=6, H=5, outliers=0, Npoints=0, Npoints_fixed=0,
            which="all", point_outliers=0, seed=3, nowarp=False, Ntri=0, tri_outliers=1, tri_only=False):
        inp, truth = synthetic.make_problem(lensmodel=lensmodel, Ncameras=Ncameras, Nframes=Nframes, W=W, H=H,
                                        seed=seed, pixel_noise=0.3, which=which, Npoints=Npoints,
                                        Npoints_fixed=Npoints_fixed)
        inp["calobject_warp"] = np.array((1e-3, -2e-3))   # away from 0 so its gradient is exercised
        if nowarp:
            del inp["calobject_warp"]
            inp["do_optimize_calobject_warp"] = False
        if sel is not None:
            inp.update(sel)
        if outliers:
            _mark_outliers(inp, outliers, seed)
        if point_outliers:
            # both flavours of "outlier" for points: weight <0 and weight ==0 (mrcal.c:4918)
            inp["observations_point"][:point_outliers, 2] = np.array((-1., 0.))[np.arange(point_outliers) % 2]
        if Ntri:
            add_triangulated_points(inp, truth, Ntri, seed + 100, outliers=tri_outliers)
            if tri_only:
                # no boards, no discrete points: the extrinsics are the whole state
                for k in ("observations_board", "indices_frame_camintrinsics_camextrinsics", "rt_ref_frame", "calobject_warp",
                          "observations_point", "indices_point_camintrinsics_camextrinsics", "points", "Npoints_fixed"):
                    inp.pop(k, None)
        cases.append((name, inp))

    for lm, tag in (("LENSMODEL_PINHOLE", "pinhole"), ("LENSMODEL_STEREOGRAPHIC", "stereographic"),
                    ("LENSMODEL_LONLAT", "lonlat"), ("LENSMODEL_LATLON", "latlon"),
                    ("LENSMODEL_OPENCV4", "opencv4"), ("LENSMODEL_OPENCV5", "opencv5"),
                    ("LENSMODEL_OPENCV8", "opencv8"), ("LENSMODEL_OPENCV12", "opencv12"),
                    ("LENSMODEL_CAHVOR", "cahvor"), ("LENSMODEL_CAHVORE_linearity=0.37", "cahvore")):
        add(f"{tag}_2cam_all", lm, 2, 4, _sel(True, True, True, True, True))
    add("splined3_2cam_corelocked", SPL3, 2, 4, _sel(False, True, True, True, True), outliers=7)
    add("splined3_3cam_all", SPL3, 3, 3, _sel(True, True, True, True, True), which="some")
    add("splined2_2cam_corelocked", SPL2, 2, 4, _sel(False, True, True, True, True), outliers=5)
    add("splined2_2cam_coreonly", SPL2, 2, 3, _sel(True, False, True, True, False))
    add("opencv8_1cam", "LENSMODEL_OPENCV8", 1, 5, _sel(True, True, False, True, True))
    add("opencv8_intrinsics_only", "LENSMODEL_OPENCV8", 2, 3, _sel(True, True, False, False, False))
    add("opencv8_frames_only", "LENSMODEL_OPENCV8", 2, 3, _sel(False, False, False, True, False))
    add("opencv8_extrinsics_warp", "LENSMODEL_OPENCV8", 3, 3, _sel(False, False, True, False, True, reg=False))
    add("opencv4_unity", "LENSMODEL_OPENCV4", 3, 3, _sel(True, True, True, True, True, unity=True), outliers=4)
    add("opencv8_noreg_outliers", "LENSMODEL_OPENCV8", 2, 4, _sel(True, True, True, True, True, reg=False), outliers=9)
    add("opencv8_nowarp_input", "LENSMODEL_OPENCV8", 2, 3, _sel(True, True, True, True, False), nowarp=True)
    add("opencv8_points", "LENSMODEL_OPENCV8", 2, 3, _sel(True, True, True, True, True), Npoints=7, point_outliers=2)
    add("opencv8_points_fixed", "LENSMODEL_OPENCV8", 3, 3, _sel(True, True, True, True, True), Npoints=8,
        Npoints_fixed=3, which="some")
    add("splined3_points", SPL3, 2, 3, _sel(False, True, True, True, True), Npoints=6, point_outliers=1)
    add("splined3_points_core", SPL3, 2, 3, _sel(True, True, True, True, True), Npoints=6, Npoints_fixed=2,
        point_outliers=2)
    add("pinhole_points_noframes", "LENSMODEL_PINHOLE", 2, 3, _sel(True, False, True, False, False), Npoints=5)
    add("cahvor_points", "LENSMODEL_CAHVOR", 3, 3, _sel(True, True, True, True, True), Npoints=6, Npoints_fixed=1,
        outliers=3, which="some")
    add("cahvore_points", "LENSMODEL_CAHVORE_linearity=-0.25", 3, 3, _sel(True, True, True, True, True), Npoints=6, Npoints_fixed=1,
        outliers=3, which="some")
    add("cahvore_lin0_coreonly", "LENSMODEL_CAHVORE_linearity=0.00", 2, 3, _sel(True, False, True, True, True))
    # triangulated points: intrinsics locked, extrinsics in the state (mrcal.c:6260-6275)
    add("tri_pinhole_only", "LENSMODEL_PINHOLE", 3, 2, _sel(False, False, True, False, False), Ntri=7, tri_only=True)
    add("tri_latlon_only", "LENSMODEL_LATLON", 2, 2, _sel(False, False, True, False, False), Ntri=5, tri_only=True, tri_outliers=0)
    add("tri_opencv4_boards_points", "LENSMODEL_OPENCV4", 3, 3, _sel(False, False, True, True, True), Npoints=5,
        Npoints_fixed=1, Ntri=6, tri_outliers=2, outliers=3)
    add("tri_pinhole_unity_only", "LENSMODEL_PINHOLE", 3, 2, _sel(False, False, True, False, False, unity=True), Ntri=20,
        tri_only=True)
    add("tri_stereographic_unity", "LENSMODEL_STEREOGRAPHIC", 3, 3, _sel(False, False, True, True, False, unity=True), Ntri=4)
    return cases


def oracle_golden(group):
    """What the compiled reference computed for the inputs of one test module (tests/golden/make_oracle_golden.py)."""
    return np.load(os.path.join(GOLDEN, f"oracle_{group}.npz"))


def layout_numbers(P):
    """A fixed list of layout integers for an oracle Problem (oracle/ref.py)."""
    out = [P.num_states(), P.num_measurements(), P.num_j_nonzero()]
    for what in ("intrinsics", "extrinsics", "frames", "points", "calobject_warp"):
        out.append(P.num_states_of(what))
    for what, i in (("intrinsics", 0), ("intrinsics", 1), ("extrinsics", 0), ("extrinsics", 1), ("frames", 0),
                    ("frames", 2), ("points", 0), ("points", 3), ("calobject_warp", 0)):
        out.append(P.state_index(what, i))
    for what, i in (("boards", 0), ("boards", 2), ("points", 0), ("points", 1), ("regularization", 0)):
        out.append(P.measurement_index(what, i))
    for what in ("boards", "points", "regularization"):
        out.append(P.num_measurements_of(what))
    return out


def inject_gross_outliers(inp, fraction, seed, shift=25.):
    """Moves a fraction of the board corners by `shift` pixels (as test-basic-calibration.py:91-100 does with its
    x20 noise), so that outlier rejection has something to find."""
    rng = np.random.default_rng(seed)
    flat = inp["observations_board"].reshape(-1, 3)
    n = max(1, int(fraction * flat.shape[0]))
    i = rng.choice(flat.shape[0], n, replace=False)
    ang = rng.uniform(0, 2 * np.pi, n)
    flat[i, 0] += shift * np.cos(ang)
    flat[i, 1] += shift * np.sin(ang)
    return inp


def solve_cases():
    """(name, optimization_inputs) whose SOLUTIONS by the reference's own mrcal_optimize() (on the restated
    libdogleg, oracle/port/dogleg_port.c) are stored in tests/golden/solve_cases.npz by
    tests/golden/make_solve_golden.py. BASELINE configs 1-3 exactly as bench.py builds them, the same with
    gross outliers and outlier rejection on, and small problems that exercise points and triangulated
    points in the outer loop."""
    cases = []
    for cfg in (1, 2, 3):
        kw, _ = synthetic.baseline_config(cfg, pixel_noise=0.3)
        cases.append((f"baseline{cfg}", kw))
    for cfg, frac in ((1, 0.01), (2, 0.005)):
        kw, _ = synthetic.baseline_config(cfg, pixel_noise=0.3)
        inject_gross_outliers(kw, frac, 100 + cfg)
        kw["do_apply_outlier_rejection"] = True
        cases.append((f"baseline{cfg}_outliers", kw))
    kw, _ = synthetic.make_problem(lensmodel=SPL3, Ncameras=2, Nframes=30, W=6, H=5, seed=11, pixel_noise=0.2)
    inject_gross_outliers(kw, 0.01, 7)
    kw["do_apply_outlier_rejection"] = True
    cases.append(("splined3_outliers", kw))
    kw, _ = synthetic.make_problem(lensmodel="LENSMODEL_OPENCV4", Ncameras=3, Nframes=8, W=6, H=5, seed=4,
                                   pixel_noise=0.2, Npoints=12, Npoints_fixed=3, which="some")
    inject_gross_outliers(kw, 0.02, 8)
    kw["do_apply_outlier_rejection"] = True
    cases.append(("opencv4_points_outliers", kw))
    # triangulated points (intrinsics locked): the outlier loop has a triangulated branch too (mrcal.c:4150-4400)
    for name in ("tri_pinhole_unity_only", "tri_opencv4_boards_points", "tri_stereographic_unity"):
        kw = dict(dict(golden_cases())[name])
        kw = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in kw.items()}
        kw["do_apply_outlier_rejection"] = True
        cases.append((name + "_rejection", kw))
    # ... and one where that branch has work to do: two observations moved far enough that their rays diverge or
    # their residual is many sigma out
    inp, truth = synthetic.make_problem(lensmodel="LENSMODEL_PINHOLE", Ncameras=3, Nframes=2, W=6, H=5, seed=5, pixel_noise=0.3)
    inp.update(_sel(False, False, True, False, False, unity=True))   # the scale of a points-only solve is free otherwise
    add_triangulated_points(inp, truth, 40, 77, outliers=0)
    for k in ("observations_board", "indices_frame_camintrinsics_camextrinsics", "rt_ref_frame", "calobject_warp"):
        inp.pop(k, None)
    inp["do_optimize_calobject_warp"] = False
    o = inp["observations_point_triangulated"]
    o[5, 0] += 900.; o[17, 1] -= 40.; o[60, 0] -= 25.
    inp["do_apply_outlier_rejection"] = True
    cases.append(("tri_divergent_rejection", inp))
    return cases
