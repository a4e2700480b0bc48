"""The N>1 path on CPU: two processes over gloo. Checks the host-side sharding
(mrcal_b200/distributed.py) and, with the compiled reference as the cost function, the
ALGORITHM of the sharded solve: the per-rank Schur-reduced normal equations, summed with
an all-reduce, equal the reduced normal equations of the whole problem (SURVEY.md 8e).
The reduced systems of the reference's Jacobians are stored under tests/golden/ for the
shards shard_inputs() makes today; a digest of each shard's inputs ties them together."""
import hashlib
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
WORLD = 2


def problem():
    from mrcal_b200 import synthetic
    kw, _ = synthetic.make_problem(lensmodel="LENSMODEL_OPENCV4", Ncameras=3, Nframes=9, W=5, H=4, seed=4,
                                   pixel_noise=0.2, Npoints=10, Npoints_fixed=2, which="some")
    return kw


def digest(kw):
    h = hashlib.sha256()
    for k in sorted(kw):
        v = kw[k]
        h.update(k.encode())
        if isinstance(v, np.ndarray):
            h.update(f"{v.dtype.str}{v.shape}".encode())
            h.update(np.ascontiguousarray(v).tobytes())
        else:
            h.update(repr(v).encode())
    return h.hexdigest()


def _reduced(J, x, e0, e1):
    Jd = J.toarray()
    H, g = Jd.T @ Jd, Jd.T @ x
    n = H.shape[0]
    sh, el = np.r_[0:e0, e1:n], np.r_[e0:e1]
    A, B, D = H[np.ix_(sh, sh)], H[np.ix_(sh, el)], H[np.ix_(el, el)]
    Dinv = np.linalg.inv(D)
    # S is a difference of nearly equal terms: its achievable accuracy is relative to |A|
    return A - B @ Dinv @ B.T, g[sh] - B @ Dinv @ g[el], np.abs(A).max(), np.abs(g).max()


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import mrcal_b200
        import problems
        from mrcal_b200 import distributed
        gold = problems.oracle_golden("distributed")
        kw = problem()
        kw_local, shard = distributed.shard_inputs(kw, rank, world)
        # the stored reduced systems are those of exactly these shards
        assert digest(kw_local) == str(gold[f"rank{rank}/digest"])
        # 1. the local slice is a valid problem by the reference's own rules (mrcal-pywrap.c:976-1244)
        I = mrcal_b200.api._Inputs(dict(kw_local))
        # 2. shards tile the frames and the observations
        t = torch.tensor([shard["f0"], shard["f1"], I.Nobs_board, I.Nobs_point, I.Nframes, I.Npoints - I.Npoints_fixed])
        ts = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(ts, t)
        ts = torch.stack(ts).numpy()
        assert ts[0, 0] == 0 and ts[-1, 1] == kw["rt_ref_frame"].shape[0] and (ts[1:, 0] == ts[:-1, 1]).all()
        assert ts[:, 2].sum() == kw["observations_board"].shape[0]
        assert ts[:, 3].sum() == kw["observations_point"].shape[0]
        assert ts[:, 4].sum() == kw["rt_ref_frame"].shape[0]
        assert ts[:, 5].sum() == kw["points"].shape[0] - 2
        # 3. the shared unknowns are laid out identically on every rank, by the reference and by the product
        n_shared = int(gold[f"rank{rank}/n_shared"])
        assert n_shared == (mrcal_b200.num_states(**kw_local) - mrcal_b200.num_states_frames(**kw_local)
                            - mrcal_b200.num_states_points(**kw_local))
        tt = torch.tensor([n_shared]); tts = [torch.zeros_like(tt) for _ in range(world)]
        dist.all_gather(tts, tt)
        assert all(int(v) == n_shared for v in tts)
        # 4. sum over ranks of the locally reduced systems == the reduced system of the whole problem.
        #    Regularization rows are replicated: only rank 0 counts them (_reduced() of the reference's J)
        St, gt = torch.from_numpy(gold[f"rank{rank}/S"].copy()), torch.from_numpy(gold[f"rank{rank}/g"].copy())
        dist.all_reduce(St)
        dist.all_reduce(gt)
        Sg, gg = gold["global/S"], gold["global/g"]
        scaleA, scaleg = gold["global/scales"]
        assert np.abs(St.numpy() - Sg).max() <= 1e-9 * scaleA
        assert np.abs(gt.numpy() - gg).max() <= 1e-9 * scaleg
        q.put((rank, "ok"))
    except Exception as e:   # pragma: no cover
        import traceback
        q.put((rank, traceback.format_exc()))
    finally:
        dist.destroy_process_group()


def test_sharding_two_ranks_gloo():
    world = WORLD
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 400)
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=180) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
    for rank, msg in results:
        assert msg == "ok", f"rank {rank}: {msg}"


def test_shard_inputs_single_rank_is_identity():
    sys.path.insert(0, ROOT)
    from mrcal_b200 import distributed, synthetic
    kw, _ = synthetic.make_problem(Ncameras=2, Nframes=5, W=4, H=4)
    loc, shard = distributed.shard_inputs(kw, 0, 1)
    assert (shard["f0"], shard["f1"]) == (0, 5)
    assert np.array_equal(loc["observations_board"], kw["observations_board"])
    assert np.array_equal(loc["indices_frame_camintrinsics_camextrinsics"], kw["indices_frame_camintrinsics_camextrinsics"])
    with pytest.raises(RuntimeError):
        distributed.shard_inputs(kw, 0, 6)
