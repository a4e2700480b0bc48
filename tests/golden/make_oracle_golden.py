#!/usr/bin/env python3
"""Builds tests/golden/oracle_*.npz: what the compiled reference (oracle/_ref) and the numpy restatement of its
solver (oracle/dogleg_np.py) return for the inputs the tests compare the product with. The tests read these files
instead of calling the oracle, so they run wherever the repository is, without the reference sources.

Needs oracle/_ref/libmrcal_ref.so, which `make -C oracle ref REF=<reference tree>` builds:

    python tests/golden/make_oracle_golden.py [group ...]

Groups (one file each): layout, cameramodel, precision, distributed, cross_reprojection, project, callback, optimize.
Every input is rebuilt from seeds by the tests' own helpers, so the stored numbers and the tests cannot drift apart
without the digests or shapes stored next to them noticing. Large outputs are sampled at fixed, seeded indices."""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.abspath(os.path.join(HERE, "..", ".."))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import ref  # noqa: E402
import problems  # noqa: E402
from mrcal_b200 import synthetic  # noqa: E402


def _clone(kw):
    return {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in kw.items()}


def layout():
    import test_layout as t
    out = {}
    for i, name in enumerate(t.LENSMODELS):
        a = ref.lensmodel_from_name(name)
        buf = C.create_string_buffer(256)
        ref.lib().mrcal_lensmodel_name(buf, 256, C.byref(a))
        out[f"lensmodel{i}/name"] = np.array(name)
        out[f"lensmodel{i}/struct"] = np.frombuffer(bytes(a), np.uint8)
        out[f"lensmodel{i}/num_params"] = np.array(ref.lensmodel_num_params(name))
        out[f"lensmodel{i}/written_name"] = np.array(buf.value.decode())
    for i, bad in enumerate(t.BAD_LENSMODELS):
        ra = ref.Lensmodel()
        ok = ref.lib().mrcal_lensmodel_from_name(C.byref(ra), bad.encode())
        out[f"bad{i}"] = np.array([bool(ok), ra.type, ref.lib().mrcal_lensmodel_type_from_name(bad.encode())])

    class Pre(C.Structure):
        _fields_ = [("ready", C.c_bool), ("segments_per_u", C.c_double)]
    for i, name in enumerate(t.PRECOMPUTED_LENSMODELS):
        a = Pre()
        ref.lib()._mrcal_precompute_lensmodel_data(C.byref(a), C.byref(ref.lensmodel_from_name(name)))
        out[f"precomputed{i}"] = np.array([float(a.ready), a.segments_per_u])
    for i, name in enumerate(t.SPLINED):
        Nx, Ny = (int(s.split("=")[1]) for s in name.split("_")[4:6])
        rx, ry = np.zeros(Nx), np.zeros(Ny)
        ref.lib().mrcal_knots_for_splined_models(rx.ctypes.data_as(C.c_void_p), ry.ctypes.data_as(C.c_void_p),
                                                 C.byref(ref.lensmodel_from_name(name)))
        out[f"knots{i}/x"], out[f"knots{i}/y"] = rx, ry
    out["grid"] = np.array([problems.layout_numbers(ref.Problem(kw)) for _, kw in t.layout_grid()], np.int32)
    for name, kw in problems.golden_cases():
        P = ref.Problem(kw)
        scale = np.ones(P.num_states())
        P.unpack_vector(scale)
        # pack divides by the scale and unpack multiplies by it: the test can restate both from the scales
        b = np.random.default_rng(1).normal(size=(3, len(scale)))
        packed = P.pack_vector(b.copy())
        assert np.array_equal(packed, b / scale) and np.array_equal(P.unpack_vector(packed.copy()), packed * scale)
        out[f"{name}/state_scale"] = scale
    for name in t.TRIANGULATED_CASES:
        P = ref.Problem(dict(problems.golden_cases())[name])
        out[f"{name}/num_measurements"] = np.array([P.num_measurements(), P.num_j_nonzero()])
    return out


def cameramodel():
    import test_cameramodel as t
    rt = t.inverse_pose_inputs()
    return {"rt": rt, "inverted": np.array([ref.invert_rt(r) for r in rt])}


def precision():
    import test_triangulated_precision as t
    L = ref.lib()
    L._mrcal_triangulated_error.restype = C.c_double
    out = []
    for c in t._cases():
        dv1, dt = (C.c_double * 3)(), (C.c_double * 3)()
        v0, v1, tt = (C.c_double * 3)(*c[0:3]), (C.c_double * 3)(*c[3:6]), (C.c_double * 3)(*c[6:9])
        e = L._mrcal_triangulated_error(dv1, dt, v0, v1, tt)
        out.append([e] + list(dv1) + list(dt))
    return {"cases": t._cases(), "error_gradient": np.array(out)}


def _reduced_of(kw, drop_regularization):
    """Schur-reduced normal equations of the reference's J (test_distributed_cpu._reduced) and the number of
    shared unknowns."""
    import test_distributed_cpu as t
    P = ref.Problem(kw)
    b, x, J = P.callback()
    nreg = P.num_measurements_of("regularization")
    if drop_regularization and nreg:
        J, x = J[:-nreg], x[:-nreg]
    e0 = P.state_index("frames", 0)
    e1 = e0 + P.num_states_of("frames") + P.num_states_of("points")
    S, g, scaleA, scaleg = t._reduced(J, x, e0, e1)
    return S, g, np.array([scaleA, scaleg]), P.num_states() - P.num_states_of("frames") - P.num_states_of("points")


def distributed():
    import test_distributed_cpu as t
    from mrcal_b200 import distributed as d
    kw = t.problem()
    out = {}
    for rank in range(t.WORLD):
        kw_local, _ = d.shard_inputs(kw, rank, t.WORLD)
        S, g, _, n_shared = _reduced_of(kw_local, rank != 0)
        out[f"rank{rank}/digest"] = np.array(t.digest(kw_local))
        out[f"rank{rank}/S"], out[f"rank{rank}/g"], out[f"rank{rank}/n_shared"] = S, g, np.array(n_shared)
    out["global/S"], out["global/g"], out["global/scales"], _ = _reduced_of(kw, False)
    return out


def cross_reprojection():
    import test_cross_reprojection_gpu as tg
    import test_cross_reprojection_oracle as to
    out = {}
    for lensmodel in to.LENSMODELS:
        kw = to.problem(lensmodel)
        P = ref.Problem(kw)
        K, b, J = P.drt_cross_reprojection__dbpacked(-1)
        i_f0, i_cw = P.state_index("frames", 0), P.state_index("calobject_warp")
        nobs = P.num_measurements_of("boards")
        cols = np.r_[i_f0:i_f0 + 6 * P.Nframes, i_cw:i_cw + 2]
        J_cols = J[:nobs].toarray()[:, cols]
        out[f"definition/{lensmodel}/K"], out[f"definition/{lensmodel}/b"] = K, b
        out[f"definition/{lensmodel}/J_cols_gram"] = J_cols.T @ J_cols
        out[f"definition/{lensmodel}/layout"] = np.array([i_f0, i_cw, nobs, P.Nframes])
    for case, (kw, icams) in tg.cases().items():
        P = ref.Problem(_clone(kw))
        for icam in icams:
            out[f"{case}/{icam}"] = P.drt_cross_reprojection__dbpacked(icam)[0]
    kw = tg.refused_problem()
    try:
        ref.Problem(_clone(kw)).drt_cross_reprojection__dbpacked(-1)
        out["refused"] = np.array(False)
    except RuntimeError:
        out["refused"] = np.array(True)
    return out


def project():
    import test_project_gpu as t
    out = {}
    for lm in t.MODELS:
        intr = t.intrinsics(lm, unproject=False)
        p = t._points(40, 1)
        q, g = ref.project(p, lm, intr, gradients=True)
        _, g3, gi = ref.project_with_intrinsics_gradient(p, lm, intr)
        out[f"{lm}/q"], out[f"{lm}/dq_dp"], out[f"{lm}/dq_dp_with_intrinsics"], out[f"{lm}/dq_dintrinsics"] = q, g, g3, gi
        intr = t.intrinsics(lm, unproject=True)
        q = ref.project(t._points(40, 2), lm, intr)
        out[f"{lm}/unproject_q"], out[f"{lm}/unproject_v"] = q, ref.unproject(q, lm, intr)
    return out


def callback():
    import test_callback_gpu as t
    out = {}
    for config in t.BASELINE_CONFIGS:
        kw, _ = synthetic.baseline_config(config)
        b, x, J = ref.Problem(kw).callback()
        out[f"config{config}/shape"] = np.array([len(b), len(x), J.nnz])
        out[f"config{config}/structure_sha256"] = np.array(t.structure_digest(J.indptr, J.indices))
        for what, v in (("b", b), ("x", x), ("Jx", J.data)):
            i = t.sample_indices(len(v))
            out[f"config{config}/{what}_index"], out[f"config{config}/{what}"] = i, v[i]
    return out


def optimize():
    import test_optimize_gpu as t
    from oracle import dogleg_np
    out = {}
    for case, kw in t.cases().items():
        r = dogleg_np.optimize(_clone(kw))
        P = r["problem"]
        out[f"{case}/b_packed"] = r["b_packed"]
        out[f"{case}/scalars"] = np.array([r["rms_reproj_error__pixels"], r["norm2_x"]])
        out[f"{case}/counts"] = np.array([r["Noutliers_board"], r["passes"]])
        for name in t.STATE_ARRAYS:
            a = getattr(P, name)
            if a is not None and a.size:
                out[f"{case}/{name}"] = a
        if P.Nobs_board:
            out[f"{case}/outliers_board"] = np.flatnonzero(P.observations_board.reshape(-1, 3)[:, 2] < 0).astype(np.int32)
    for lensmodel, kw in t.tight_cases().items():
        r = dogleg_np.optimize(_clone(kw), **t.TIGHT)
        out[f"tight/{lensmodel}/b_packed"] = r["b_packed"]
        out[f"tight/{lensmodel}/norm2_x"] = np.array(r["norm2_x"])
    return out


GROUPS = dict(layout=layout, cameramodel=cameramodel, precision=precision, distributed=distributed,
              cross_reprojection=cross_reprojection, project=project, callback=callback, optimize=optimize)


def main():
    if not ref.available():
        sys.exit(f"{ref.LIBPATH} is missing: build it with make -C oracle ref REF=<reference tree>")
    for group in sys.argv[1:] or GROUPS:
        data = GROUPS[group]()
        path = os.path.join(HERE, f"oracle_{group}.npz")
        np.savez_compressed(path, **data)
        print(f"{path}: {len(data)} arrays, {os.path.getsize(path)} bytes", flush=True)


if __name__ == "__main__":
    main()
