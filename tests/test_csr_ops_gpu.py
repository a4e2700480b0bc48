"""_Jt_x / _A_Jt_J_At / _A_Jt_J_At__2 on the GPU (mrcal_b200/csrc/csr_ops.cu) against the loops of the reference's
numpysane wrappers (mrcal-genpywrap.py:477-731), restated here in numpy."""
import numpy as np
import pytest
import scipy.sparse

pytestmark = pytest.mark.gpu


def _random_csr(rng, Nrows, Ncols, density):
    J = scipy.sparse.random(Nrows, Ncols, density=density, format="csr", random_state=np.random.RandomState(rng.integers(1 << 30)))
    J.sort_indices()
    return J.indptr.astype(np.int32), J.indices.astype(np.int32), J.data.astype(np.float64), J


def test_Jt_x_bit_identical_to_the_reference_loop():
    import mrcal_b200
    rng = np.random.default_rng(0)
    Jp, Ji, Jx, J = _random_csr(rng, 5000, 300, 0.03)
    x = rng.normal(size=5000)
    out = np.zeros(300)
    mrcal_b200._Jt_x(Jp, Ji, Jx, x, out=out)
    # the reference's loop: rows in order, y[icol] += j*x[irow]
    y = np.zeros(300)
    for r in range(5000):
        for e in range(Jp[r], Jp[r + 1]):
            y[Ji[e]] += Jx[e] * x[r]
    assert np.array_equal(out, y)
    with pytest.raises(RuntimeError):
        mrcal_b200._Jt_x(Jp, Ji, Jx, x[:-1], out=out)


@pytest.mark.parametrize("Nx", [2, 3, 7])
def test_A_Jt_J_At(Nx):
    import mrcal_b200
    rng = np.random.default_rng(Nx)
    Jp, Ji, Jx, J = _random_csr(rng, 9000, 200, 0.05)
    A = rng.normal(size=(4, Nx, 200))          # broadcast over the leading dimension
    Nlead = 7001
    got = mrcal_b200._A_Jt_J_At(A, Jp, Ji, Jx, Nleading_rows_J=Nlead)
    Jl = J[:Nlead].toarray()
    ref = np.einsum("bik,rk,rl,bjl->bij", A, Jl, Jl, A)
    assert got.shape == (4, Nx, Nx)
    assert np.abs(got - ref).max() <= 1e-12 * np.abs(ref).max()
    assert np.array_equal(got, np.swapaxes(got, -1, -2))
    if Nx == 2:
        assert np.array_equal(mrcal_b200._A_Jt_J_At__2(A, Jp, Ji, Jx, Nleading_rows_J=Nlead), got)
    with pytest.raises(RuntimeError):
        mrcal_b200._A_Jt_J_At(A, Jp, Ji, Jx)


def test_on_a_calibration_jacobian():
    """The shapes the uncertainty code uses: J of a calibration problem, A = 2 x Nstate, board rows only."""
    import mrcal_b200
    from mrcal_b200 import synthetic
    kw, _ = synthetic.make_problem(lensmodel="LENSMODEL_OPENCV8", Ncameras=2, Nframes=20, W=10, H=10, seed=1, pixel_noise=0.3)
    b, x, J, _ = mrcal_b200.optimizer_callback(**kw, no_factorization=True)
    Nboards = mrcal_b200.num_measurements_boards(**kw)
    rng = np.random.default_rng(3)
    A = rng.normal(size=(2, J.shape[1]))
    got = mrcal_b200._A_Jt_J_At__2(A, J.indptr, J.indices, J.data, Nleading_rows_J=Nboards)
    JA = J[:Nboards] @ A.T
    assert np.abs(got - JA.T @ JA).max() <= 1e-12 * np.abs(JA.T @ JA).max()
    out = np.zeros(J.shape[1])
    mrcal_b200._Jt_x(J.indptr, J.indices, J.data, x, out=out)
    assert np.abs(out - J.T @ x).max() <= 1e-12 * np.abs(J.T @ x).max()
