"""GPU parity tests (run with -m gpu on a B200): the CUDA path through the C ABI vs the CPU oracle on the same
seeded inputs, vs the committed golden vectors (outputs of the reference's own code), and -- at the BASELINE
C2 size -- through size-independent properties (linearity, symmetry, row extraction, noise shift).

Stated tolerances (fp32 path; oracle evaluated in fp64):
  fused K.V            rel-l2 <= 5e-6 (tcgen05, 3xTF32 split) / 2e-6 (simt)
  kernel entries       abs   <= 2e-6 vs the reference-generated golden matrices (fp32 goldens: 1e-5)
  pivoted Cholesky     pivots bit-exact (integer work); L rel-l2 <= 1e-5
  preconditioned mBCG  same iteration count; solves rel <= 5e-4; tridiagonals rel <= 1e-4; inv_quad rel <= 1e-4;
                       log-det (identical probes + preconditioner) rel <= 1e-4
  MLL                  |gpu - oracle| <= 1e-4 |oracle| and within 2 % of dense Cholesky
"""
import math
import warnings

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import kernels as ok, linalg as ol, mll as om  # noqa: E402

BACKENDS = ["tcgen05", "simt"]
KV_TOL = {"tcgen05": 5e-6, "simt": 2e-6}


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-300)).item()


@pytest.fixture(scope="module")
def Plan(cuda_dev):
    from gpytorch_b200.engine import Plan as P

    return P


# ---------------------------------------------------------------------------------------------------------
# kernel seam
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("kind", ["rbf", "matern12", "matern32", "matern52"])
def test_kmv_matches_oracle(Plan, cuda_dev, backend, kind):
    g = torch.Generator().manual_seed(11)
    n, d, t = 1500, 7, 11
    x = torch.rand(n, d, generator=g, dtype=torch.float64)
    v = torch.randn(n, t, generator=g, dtype=torch.float64)
    K = ok.kernel_matrix(kind, x, x, 0.9, 1.7, True)
    p = Plan(x.float().to(cuda_dev), backend=backend).set_hypers(kind, 0.9, 1.7, 0.3)
    assert p.info()["backend"] == backend
    assert rel(p.kmv(v.float().to(cuda_dev)), K @ v) < KV_TOL[backend]
    assert rel(p.kmv(v.float().to(cuda_dev), add_noise=True), K @ v + 0.3 * v) < KV_TOL[backend]
    p.close()


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("n1,n2,d,t", [(1, 1, 1, 1), (127, 95, 3, 1), (129, 97, 10, 16), (777, 1300, 10, 5), (300, 40, 20, 33), (64, 2000, 41, 3)])
def test_kmv_ragged_shapes_cross_covariance(Plan, cuda_dev, backend, n1, n2, d, t):
    g = torch.Generator().manual_seed(n1 + n2)
    x1 = torch.rand(n1, d, generator=g, dtype=torch.float64)
    x2 = torch.rand(n2, d, generator=g, dtype=torch.float64)
    v = torch.randn(n2, t, generator=g, dtype=torch.float64)
    K = ok.kernel_matrix("matern52", x1, x2, 1.3, 0.8, False)
    p = Plan(x1.float().to(cuda_dev), x2.float().to(cuda_dev), backend=backend).set_hypers("matern52", 1.3, 0.8, 0.1)
    out = p.kmv(v.float().to(cuda_dev))
    assert out.shape == (n1, t)
    assert rel(out, K @ v) < 2 * KV_TOL[backend]
    p.close()


@pytest.mark.parametrize("backend", BACKENDS)
def test_kmv_ard_lengthscales(Plan, cuda_dev, backend):
    g = torch.Generator().manual_seed(5)
    n, d = 900, 6
    x = torch.rand(n, d, generator=g, dtype=torch.float64)
    v = torch.randn(n, 4, generator=g, dtype=torch.float64)
    ls = torch.linspace(0.5, 1.5, d, dtype=torch.float64)
    K = ok.kernel_matrix("rbf", x, x, ls, 1.0, True)
    p = Plan(x.float().to(cuda_dev), backend=backend).set_hypers("rbf", ls.tolist(), 1.0, 0.0)
    assert rel(p.kmv(v.float().to(cuda_dev)), K @ v) < KV_TOL[backend]
    p.close()


def test_large_d_falls_back_to_simt_and_tcgen05_refuses(Plan, cuda_dev):
    x = torch.rand(200, 60)
    p = Plan(x.to(cuda_dev), backend="auto").set_hypers("rbf", 3.0, 1.0, 0.1)
    assert p.info()["backend"] == "simt"  # 3d+4 > 128
    p.close()
    with pytest.raises(RuntimeError, match="tcgen05"):
        Plan(x.to(cuda_dev), backend="tcgen05").set_hypers("rbf", 3.0, 1.0, 0.1)


@pytest.mark.parametrize("tag", ["a", "b", "c", "d"])
def test_kernel_entries_match_reference_golden(Plan, cuda_dev, golden, tag):
    """rows() / K.V against matrices produced by the reference's own RBFCovariance / MaternCovariance (the golden file holds
    the rows `idx` of each), and against the fp64 oracle -- pinned to the same reference outputs on the CPU -- everywhere."""
    key = f"{tag}_f64"
    x1 = torch.from_numpy(golden[f"{key}_x1"])
    same = bool(golden[f"{key}_same"])
    x2 = None if same else torch.from_numpy(golden[f"{key}_x2"])
    ls = float(golden[f"{key}_ls"])
    idx = torch.from_numpy(golden[f"{key}_rows"])
    for kind, nk in (("rbf", "rbf"), ("matern12", "mat12"), ("matern32", "mat32"), ("matern52", "mat52")):
        Kgold = torch.from_numpy(golden[f"{key}_{nk}"])
        Kref = ok.kernel_matrix(kind, x1, x1 if same else x2, ls, 1.0, same)
        p = Plan(x1.float().to(cuda_dev), None if same else x2.float().to(cuda_dev), backend="simt").set_hypers(kind, ls, 1.0, 0.0)
        rows = p.rows(torch.arange(x1.size(0))).double().cpu()
        assert (rows - Kref).abs().max().item() < 2e-6
        assert (rows[idx] - Kgold).abs().max().item() < 2e-6
        p.close()
        for backend in BACKENDS:
            p = Plan(x1.float().to(cuda_dev), None if same else x2.float().to(cuda_dev), backend=backend).set_hypers(kind, ls, 1.0, 0.0)
            eye = torch.eye(Kref.size(1), dtype=torch.float32)[:, :16].contiguous()
            out = p.kmv(eye.to(cuda_dev)).double().cpu()  # K @ I[:, :16] = first 16 columns of K
            assert (out - Kref[:, :16]).abs().max().item() < 3e-6
            assert (out[idx] - Kgold[:, :16]).abs().max().item() < 3e-6
            p.close()
    # fp32 goldens: what the reference itself produces in its default dtype
    K32 = torch.from_numpy(golden[f"{tag}_f32_rbf"]).double()
    idx32 = torch.from_numpy(golden[f"{tag}_f32_rows"])
    p = Plan(torch.from_numpy(golden[f"{tag}_f32_x1"]).to(cuda_dev),
             None if same else torch.from_numpy(golden[f"{tag}_f32_x2"]).to(cuda_dev), backend="simt").set_hypers("rbf", ls, 1.0, 0.0)
    assert (p.rows(idx32).double().cpu() - K32).abs().max().item() < 1e-5
    p.close()


def test_rbf_known_answer_through_api(cuda_dev):
    # /root/reference/test/kernels/test_rbf_kernel.py:126-137
    import gpytorch_b200 as gp

    a = torch.tensor([4.0, 2.0, 8.0]).view(3, 1).to(cuda_dev)
    b = torch.tensor([0.0, 2.0, 4.0]).view(3, 1).to(cuda_dev)
    kernel = gp.kernels.RBFKernel().initialize(lengthscale=2.0).to(cuda_dev)
    actual = torch.tensor([[16.0, 4, 0], [4, 0, 4], [64, 36, 16]]).mul_(-0.5).div_(4.0).exp_()
    res = kernel(a, b).to_dense().cpu()
    assert torch.norm(res - actual) < 1e-5


def test_rows_diag_and_getitem(Plan, cuda_dev):
    x = torch.rand(500, 4, dtype=torch.float64, generator=torch.Generator().manual_seed(2))
    K = ok.kernel_matrix("matern32", x, x, 0.8, 2.0, True)
    p = Plan(x.float().to(cuda_dev)).set_hypers("matern32", 0.8, 2.0, 0.1)
    idx = torch.tensor([0, 5, 499, 17, 17])
    assert rel(p.rows(idx), K[idx]) < 2e-6
    assert torch.equal(p.diag().cpu(), torch.full((500,), 2.0))
    p.close()


# ---------------------------------------------------------------------------------------------------------
# solver seam
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d,kind,ls,rank", [(1000, 3, "rbf", 0.5, 15), (3000, 10, "rbf", 1.0, 100), (2000, 4, "matern52", 0.7, 50)])
def test_pivoted_cholesky_bit_exact_pivots_and_preconditioner(Plan, cuda_dev, n, d, kind, ls, rank):
    x, y = om.synthetic_problem(n, d, 0, torch.float64)
    K = ok.kernel_matrix(kind, x, x, ls, 1.0, True)
    Lo, pivo = ol.pivoted_cholesky(torch.ones(n, dtype=torch.float64), lambda i: K[i], rank, 1e-3)
    p = Plan(x.float().to(cuda_dev)).set_hypers(kind, ls, 1.0, 0.1)
    lt, piv, st = p.pivoted_cholesky(rank, 1e-3)
    assert st == 0 and lt.size(0) == Lo.size(1)
    assert piv.cpu().tolist() == pivo.tolist()  # integer / index work: bit exact
    assert rel(lt.t(), Lo) < 1e-5
    pre = ol.build_preconditioner(Lo, 0.1, pivo)
    w, logdet, _ = p.precond_build(lt)
    assert logdet == pytest.approx(pre.logdet, rel=1e-6)
    v = torch.randn(n, 4, dtype=torch.float64)
    wd = w.double().cpu()
    assert rel((v - wd @ (wd.t() @ v)) / 0.1, pre.apply(v)) < 1e-5
    eps1, eps2, _ = om.make_probe_noise(n, lt.size(0), 10, 1)
    z = p.precond_probes(lt, eps1.to(cuda_dev), eps2.to(cuda_dev))
    assert rel(z, pre.probes(eps1.double()[: Lo.size(1)], eps2.double())) < 1e-5
    p.close()


def test_pivoted_cholesky_stops_on_tolerance(Plan, cuda_dev):
    x, _ = om.synthetic_problem(1500, 2, 0, torch.float64)
    K = ok.kernel_matrix("rbf", x, x, 1.0, 1.0, True)  # smooth 2-D kernel: low numerical rank
    Lo, pivo = ol.pivoted_cholesky(torch.ones(1500, dtype=torch.float64), lambda i: K[i], 120, 1e-2)
    p = Plan(x.float().to(cuda_dev)).set_hypers("rbf", 1.0, 1.0, 0.1)
    lt, piv, _ = p.pivoted_cholesky(120, 1e-2)
    assert lt.size(0) == Lo.size(1) < 120
    assert piv.cpu().tolist() == pivo.tolist()
    p.close()


def test_pivoted_cholesky_persistent_and_stepwise_paths_agree(Plan, cuda_dev, monkeypatch):
    """The cooperative single-launch kernel and the one-launch-per-step fallback run the same arithmetic per entry:
    identical pivots and bit-identical factors (also with more rows than resident threads: grid-stride path)."""
    for n, d, kind, rank in ((5000, 6, "rbf", 60), (3001, 3, "matern32", 25)):
        x, _ = om.synthetic_problem(n, d, 0, torch.float32)
        p = Plan(x.to(cuda_dev)).set_hypers(kind, 0.8, 1.3, 0.1)
        monkeypatch.delenv("GP_PC_STEPWISE", raising=False)
        lt1, piv1, _ = p.pivoted_cholesky(rank, 1e-4)
        monkeypatch.setenv("GP_PC_STEPWISE", "1")
        lt2, piv2, _ = p.pivoted_cholesky(rank, 1e-4)
        monkeypatch.delenv("GP_PC_STEPWISE", raising=False)
        assert piv1.cpu().tolist() == piv2.cpu().tolist()
        assert torch.equal(lt1, lt2)
        p.close()


@pytest.mark.parametrize("backend", BACKENDS)
def test_mbcg_preconditioned_matches_oracle(Plan, cuda_dev, backend):
    n, d = 3000, 10
    x, y = om.synthetic_problem(n, d, 0, torch.float64)
    A = ok.kernel_matrix("rbf", x, x, 1.0, 1.0, True) + 0.1 * torch.eye(n, dtype=torch.float64)
    rhs = torch.randn(n, 11, generator=torch.Generator().manual_seed(5), dtype=torch.float64)
    p = Plan(x.float().to(cuda_dev), backend=backend).set_hypers("rbf", 1.0, 1.0, 0.1)
    lt, piv, _ = p.pivoted_cholesky(50, 1e-3)
    W, _, _ = p.precond_build(lt)
    pre = ol.build_preconditioner(lt.double().cpu().t().contiguous(), 0.1)
    so, to, io = ol.linear_cg(lambda v: A @ v, rhs, n_tridiag=10, preconditioner=pre.apply, return_info=True)
    sg, tg, ig = p.mbcg(rhs.float().to(cuda_dev), 10, 1.0, 1000, 20, W)
    assert ig.iters == io.iters == 21 and ig.tridiag_size == 20  # SURVEY.md Appendix A.2 stop rule
    assert rel(sg, so) < 5e-4
    assert rel(tg, to) < 1e-4
    assert p.slq_logdet(tg, n) == pytest.approx(ol.slq_logdet(to, n), rel=1e-4)
    # tighter tolerance: converges to the true solution
    sg2, _, ig2 = p.mbcg(rhs.float().to(cuda_dev), 0, 1e-4, 1000, 20, W)
    assert rel(sg2, torch.linalg.solve(A, rhs)) < 5e-4
    p.close()


def test_mbcg_unpreconditioned_early_coefficients_and_solution(Plan, cuda_dev):
    # ill-conditioned (RBF l=0.5, d=3): fp32 and fp64 Krylov recurrences diverge after a few steps -- the reference's own
    # fp32 run does too -- so compare the first coefficients and the converged solution, not every tridiagonal entry
    n = 1000
    x, y = om.synthetic_problem(n, 3, 0, torch.float64)
    A = ok.kernel_matrix("rbf", x, x, 0.5, 1.0, True) + 0.1 * torch.eye(n, dtype=torch.float64)
    rhs = torch.randn(n, 6, generator=torch.Generator().manual_seed(5), dtype=torch.float64)
    p = Plan(x.float().to(cuda_dev)).set_hypers("rbf", 0.5, 1.0, 0.1)
    so, to, io = ol.linear_cg(lambda v: A @ v, rhs, n_tridiag=6, return_info=True)
    sg, tg, ig = p.mbcg(rhs.float().to(cuda_dev), 6, 1.0, 1000, 20, None)
    assert ig.iters == 21 and tg.shape == to.shape
    assert rel(tg[:, :4, :4], to[:, :4, :4]) < 1e-3
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        sg2, _, ig2 = p.mbcg(rhs.float().to(cuda_dev), 0, 1e-3, 1000, 20, None)
    assert rel(sg2, torch.linalg.solve(A, rhs)) < 5e-3
    p.close()


def test_mbcg_zero_rhs_column_and_not_converged_warning(Plan, cuda_dev):
    from gpytorch_b200 import NumericalWarning

    n = 1200
    x, y = om.synthetic_problem(n, 3, 0, torch.float32)
    p = Plan(x.to(cuda_dev)).set_hypers("rbf", 0.5, 1.0, 0.1)
    rhs = torch.randn(n, 3)
    rhs[:, 1] = 0.0
    sol, _, info = p.mbcg(rhs.to(cuda_dev), 0, 1.0, 1000, 20, None)
    assert torch.all(sol[:, 1] == 0) and torch.isfinite(sol).all()
    with pytest.warns(NumericalWarning, match="CG terminated"):
        p.mbcg(rhs.to(cuda_dev), 0, 1e-9, 12, 10, None)
    with pytest.raises(RuntimeError, match="tridiagonalization larger"):
        p.mbcg(rhs.to(cuda_dev), 2, 1.0, 5, 20, None)
    p.close()


def test_nan_in_matmul_raises_like_the_reference(Plan, cuda_dev):
    # linear_cg: "NaNs encountered when trying to perform matrix-vector multiplication" (RuntimeError)
    n = 1500
    x, y = om.synthetic_problem(n, 3, 0, torch.float32)
    x[17, 1] = float("nan")
    p = Plan(x.to(cuda_dev)).set_hypers("rbf", 0.5, 1.0, 0.1)
    with pytest.raises(RuntimeError, match="NaNs encountered"):
        p.mbcg(torch.randn(n, 2).to(cuda_dev), 0, 1.0, 50, 20, None)
    # mean-centring (kernels/kernel.py:35-37) spreads one NaN coordinate over every entry of K
    assert torch.isnan(p.kmv(torch.randn(n, 3).to(cuda_dev))).all()
    p.close()


def test_bad_hyperparameters_are_rejected(Plan, cuda_dev):
    p = Plan(torch.rand(100, 2).to(cuda_dev))
    with pytest.raises(RuntimeError, match="positive"):
        p.set_hypers("rbf", -1.0, 1.0, 0.1)
    with pytest.raises(RuntimeError, match="does not match"):
        p.set_hypers("rbf", [1.0, 2.0, 3.0], 1.0, 0.1)
    with pytest.raises(KeyError):
        p.set_hypers("periodic", 1.0, 1.0, 0.1)
    p.close()


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("n,d,kind,ls,rank", [(3000, 10, "rbf", 1.0, 100), (2500, 6, "matern52", 1.0, 30), (2200, 4, "matern12", 0.7, 20)])
def test_mll_matches_oracle_and_cholesky(Plan, cuda_dev, backend, n, d, kind, ls, rank):
    x, y = om.synthetic_problem(n, d, 0, torch.float32)
    pn = om.make_probe_noise(n, rank, 10, 1)
    ch = om.mll_cholesky(kind, x.double(), y.double(), 0.0, ls, 1.0, 0.1)
    ro = om.mll_bbmm(kind, x.double(), y.double(), 0.0, ls, 1.0, 0.1, tuple(a.double() for a in pn), precond_size=rank)
    r32 = om.mll_bbmm(kind, x, y, 0.0, ls, 1.0, 0.1, pn, precond_size=rank)  # the reference's own default dtype
    p = Plan(x.to(cuda_dev), backend=backend).set_hypers(kind, ls, 1.0, 0.1)
    res, sol = p.mll(y.to(cuda_dev), pn[0].to(cuda_dev), pn[1].to(cuda_dev), pn[2].to(cuda_dev), 10, rank, 2000, want_solve=True)
    assert res.cg_iters == ro.iters == 21 and res.precond_rank == ro.precond.L.size(1)

    # stated tolerance: 1e-4 relative to the fp64 oracle, or -- on the less smooth / worse conditioned kernels, where
    # 21 loose CG steps amplify fp32 rounding -- no further from fp64 than 3x the fp32 run of the same reference algorithm
    def close(gpu, o64, o32):
        # Matern-1/2 is not smooth at 0: 21 loose CG steps amplify the ~5e-7 K.V differences to ~5e-4 (stated: 1e-3)
        floor = 1e-3 if kind == "matern12" else 1e-4
        return abs(gpu - o64) <= max(floor * abs(o64), 3.0 * abs(o32 - o64))

    assert close(res.inv_quad, ro.inv_quad, r32.inv_quad), (res.inv_quad, ro.inv_quad, r32.inv_quad)
    assert close(res.logdet, ro.logdet, r32.logdet), (res.logdet, ro.logdet, r32.logdet)
    assert close(res.mll, ro.mll, r32.mll)
    assert res.mll == pytest.approx(ch.mll, rel=2e-2)
    assert rel(sol, ro.solves[:, -1]) < max(1e-3, 3 * rel(r32.solves[:, -1], ro.solves[:, -1]))
    p.close()


def test_mll_no_preconditioner_branch(Plan, cuda_dev):
    # N < min_preconditioning_size: Rademacher probes, plain CG (C1-like); compare with the fp32 oracle statistics
    n = 1000
    x, y = om.synthetic_problem(n, 3, 0, torch.float32)
    pn = om.make_probe_noise(n, 15, 10, 1)
    ro = om.mll_bbmm("rbf", x, y, 0.0, 0.5, 1.0, 0.1, pn)
    ch = om.mll_cholesky("rbf", x.double(), y.double(), 0.0, 0.5, 1.0, 0.1)
    p = Plan(x.to(cuda_dev)).set_hypers("rbf", 0.5, 1.0, 0.1)
    res, _ = p.mll(y.to(cuda_dev), pn[0].to(cuda_dev), pn[1].to(cuda_dev), pn[2].to(cuda_dev), 10, 15, 2000)
    assert res.precond_rank == 0 and res.cg_iters == 21
    assert res.inv_quad == pytest.approx(ro.inv_quad, rel=2e-2)   # fp32 CG at tol=1 on an ill-conditioned system
    assert res.logdet == pytest.approx(ch.logdet, rel=2e-2)
    assert res.mll == pytest.approx(ch.mll, rel=3e-2)
    p.close()


def test_lanczos_matches_oracle(Plan, cuda_dev):
    n = 1500
    x, y = om.synthetic_problem(n, 4, 0, torch.float64)
    A = ok.kernel_matrix("rbf", x, x, 0.6, 1.0, True) + 0.1 * torch.eye(n, dtype=torch.float64)
    init = torch.randn(n, 1, dtype=torch.float64, generator=torch.Generator().manual_seed(9))
    Qo, To = ol.lanczos_tridiag(lambda v: A @ v, 30, init)
    p = Plan(x.float().to(cuda_dev)).set_hypers("rbf", 0.6, 1.0, 0.1)
    Q, T = p.lanczos(init[:, 0].float().to(cuda_dev), 30)
    assert T.shape == To[0].shape
    Qd = Q.double().cpu()
    assert (Qd.t() @ Qd - torch.eye(Qd.size(1), dtype=torch.float64)).abs().max() < 1e-5
    assert (Qd.t() @ A @ Qd - T.double().cpu()).abs().max() < 1e-3
    assert torch.allclose(torch.linalg.eigvalsh(T.double().cpu()), torch.linalg.eigvalsh(To[0]), rtol=1e-3, atol=1e-4)
    p.close()


@pytest.mark.parametrize("kind", ["rbf", "matern12", "matern32", "matern52"])
@pytest.mark.parametrize("ard", [False, True])
def test_bilinear_derivative_matches_autograd(Plan, cuda_dev, kind, ard):
    n, d, s = 800, 5, 7
    g = torch.Generator().manual_seed(2)
    x = torch.rand(n, d, generator=g, dtype=torch.float64)
    Lf = torch.randn(n, s, generator=g, dtype=torch.float64)
    Rt = torch.randn(n, s, generator=g, dtype=torch.float64)
    ls = (torch.linspace(0.6, 1.1, d, dtype=torch.float64) if ard else torch.tensor(0.8, dtype=torch.float64)).requires_grad_(True)
    os_ = torch.tensor(1.3, dtype=torch.float64, requires_grad=True)
    (Lf * (ok.kernel_matrix(kind, x, x, ls, os_, True) @ Rt)).sum().backward()
    p = Plan(x.float().to(cuda_dev)).set_hypers(kind, ls.detach().reshape(-1).tolist(), 1.3, 0.1)
    gl, go = p.bilinear_grad(Lf.float().to(cuda_dev), Rt.float().to(cuda_dev))
    assert np.allclose(gl, ls.grad.reshape(-1).numpy(), rtol=2e-4, atol=1e-2)
    assert go == pytest.approx(os_.grad.item(), rel=2e-4, abs=1e-2)
    p.close()


# ---------------------------------------------------------------------------------------------------------
# BASELINE C2 size: size-independent properties (the oracle cannot run here in seconds)
# ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def c2(Plan, cuda_dev):
    n, d = 50000, 10
    x, y = om.synthetic_problem(n, d, 0, torch.float32)
    p = Plan(x.to(cuda_dev), backend="tcgen05").set_hypers("rbf", 1.0, 1.0, 0.1)
    yield p, x, y
    p.close()


def test_c2_linearity_symmetry_rows_and_backends_agree(c2, Plan, cuda_dev):
    p, x, y = c2
    n = x.size(0)
    g = torch.Generator().manual_seed(1)
    u = torch.randn(n, 4, generator=g).to(cuda_dev)
    v = torch.randn(n, 4, generator=g).to(cuda_dev)
    Ku, Kv = p.kmv(u), p.kmv(v)
    # linearity: K(2u - 3v) = 2 Ku - 3 Kv
    assert rel(p.kmv(2 * u - 3 * v), 2 * Ku - 3 * Kv) < 1e-5
    # symmetry: <u, K v> = <K u, v>
    a = (u.double() * Kv.double()).sum(0); b = (Ku.double() * v.double()).sum(0)
    assert torch.allclose(a, b, rtol=1e-5, atol=1e-2)
    # noise shift
    assert rel(p.kmv(u, add_noise=True) - Ku, 0.1 * u) < 1e-3
    # row extraction vs the fused product on a few rows (fp64 reference on the CPU for those rows only)
    idx = torch.tensor([0, 1, 127, 128, 25000, 49999])
    rows = p.rows(idx)
    assert rel((rows.double() @ u.double()), Ku[idx.to(cuda_dev)]) < 1e-5
    Kr = ok.kernel_matrix("rbf", x[idx].double(), x.double(), 1.0, 1.0, False)
    # the oracle centres by x1's mean; stationary kernel -> identical values
    assert (rows.double().cpu() - Kr).abs().max() < 2e-6
    # the two independent kernels agree at full size
    ps = Plan(x.to(cuda_dev), backend="simt").set_hypers("rbf", 1.0, 1.0, 0.1)
    assert rel(Ku, ps.kmv(u)) < 1e-5
    ps.close()


def test_c2_mll_full_size_is_consistent(c2, cuda_dev):
    p, x, y = c2
    n = x.size(0)
    pn = om.make_probe_noise(n, 100, 10, 1)
    res, sol = p.mll(y.to(cuda_dev), pn[0].to(cuda_dev), pn[1].to(cuda_dev), pn[2].to(cuda_dev), 10, 100, 2000, want_solve=True)
    assert res.cg_iters == 21 and res.tridiag_size == 20 and res.precond_rank == 100
    # the reported CG residual is the true residual of the returned solve: |K_hat s - y| / |y| == resid[y column]
    # (cg_tolerance = 1 is loose by design: the reference trains with it)
    r = p.kmv(sol, add_noise=True) - y.to(cuda_dev)
    true_res = (r.norm() / y.norm()).item()
    assert true_res == pytest.approx(res.resid[10], rel=5e-2) and true_res < 1.0
    assert res.inv_quad == pytest.approx(float((sol.double() * y.to(cuda_dev).double()).sum()), rel=1e-6)
    assert math.isfinite(res.logdet) and -2.0 < res.mll < 2.0
    # determinism: same inputs, same bits
    res2, _ = p.mll(y.to(cuda_dev), pn[0].to(cuda_dev), pn[1].to(cuda_dev), pn[2].to(cuda_dev), 10, 100, 2000)
    assert res2.inv_quad == res.inv_quad and res2.logdet == res.logdet


def test_c4_batch_of_independent_problems(Plan, cuda_dev):
    """BASELINE config 4 (batched exact GP, independent hyper-parameters per batch element) runs as one plan per batch
    element (SURVEY.md section 2 row 18: the batch dimension of the path, not the Kronecker structure); sizes reduced so the
    fp64 oracle finishes in seconds."""
    b, n, d = 4, 2400, 8
    g = torch.Generator().manual_seed(4)
    for i in range(b):
        x = torch.rand(n, d, generator=g)
        y = torch.sin(2 * x.sum(-1)) + 0.1 * torch.randn(n, generator=g)
        ls, osc, nz = 0.8 + 0.2 * i, 1.0 + 0.5 * i, 0.05 * (i + 1)
        pn = om.make_probe_noise(n, 40, 10, 10 + i)
        ro = om.mll_bbmm("rbf", x.double(), y.double(), 0.0, ls, osc, nz, tuple(a.double() for a in pn), precond_size=40)
        r32 = om.mll_bbmm("rbf", x, y, 0.0, ls, osc, nz, pn, precond_size=40)   # the reference's default dtype
        p = Plan(x.to(cuda_dev)).set_hypers("rbf", ls, osc, nz)
        res, _ = p.mll(y.to(cuda_dev), pn[0].to(cuda_dev), pn[1].to(cuda_dev), pn[2].to(cuda_dev), 10, 40, 2000)
        assert res.cg_iters == ro.iters
        # 1e-4 of the fp64 oracle, or (element 0: noise 0.05, where the fp32 reference run itself is 1e-3 off in the
        # inverse quadratic form) no further from fp64 than 3x the fp32 run of the same algorithm; the MLL itself is a
        # near-cancelling sum (|mll| ~ 0.08 from terms of ~1), so it is bounded through its two terms
        def close(gpu, o64, o32):
            return abs(gpu - o64) <= max(1e-4 * abs(o64), 3.0 * abs(o32 - o64))
        assert close(res.inv_quad, ro.inv_quad, r32.inv_quad), (i, res.inv_quad, ro.inv_quad, r32.inv_quad)
        assert close(res.logdet, ro.logdet, r32.logdet), (i, res.logdet, ro.logdet, r32.logdet)
        bound = (max(1e-4 * abs(ro.inv_quad), 3 * abs(r32.inv_quad - ro.inv_quad))
                 + max(1e-4 * abs(ro.logdet), 3 * abs(r32.logdet - ro.logdet))) / (2 * n)
        assert abs(res.mll - ro.mll) <= bound
        p.close()


def test_c1_small_problem_through_cg_path(Plan, cuda_dev):
    """BASELINE config 1 (N=1000, d=3): below min_preconditioning_size -> Rademacher probes, plain mBCG."""
    n = 1000
    x, y = om.synthetic_problem(n, 3, 0, torch.float32)
    pn = om.make_probe_noise(n, 15, 10, 1)
    r32 = om.mll_bbmm("rbf", x, y, 0.0, 0.5, 1.0, 0.1, pn)
    for backend in BACKENDS:
        p = Plan(x.to(cuda_dev), backend=backend).set_hypers("rbf", 0.5, 1.0, 0.1)
        res, _ = p.mll(y.to(cuda_dev), pn[0].to(cuda_dev), pn[1].to(cuda_dev), pn[2].to(cuda_dev), 10, 15, 2000)
        assert res.cg_iters == r32.iters == 21 and res.precond_rank == 0 and res.tridiag_size == 20
        assert res.mll == pytest.approx(r32.mll, rel=2e-2)
        p.close()


# ---------------------------------------------------------------------------------------------------------
# the gpytorch-style public API end to end
# ---------------------------------------------------------------------------------------------------------
def _make_model(gp, x, y, kind="rbf", ard=None):
    lik = gp.likelihoods.GaussianLikelihood()
    base = gp.kernels.RBFKernel(ard_num_dims=ard) if kind == "rbf" else gp.kernels.MaternKernel(nu=2.5, ard_num_dims=ard)

    class M(gp.models.ExactGP):
        def __init__(self):
            super().__init__(x, y, lik)
            self.mean_module = gp.means.ConstantMean()
            self.covar_module = gp.kernels.ScaleKernel(base)

        def forward(self, xx):
            return gp.distributions.MultivariateNormal(self.mean_module(xx), self.covar_module(xx))

    m = M().to(x.device)
    return m, lik.to(x.device)


def test_api_mll_forward_backward_vs_dense_autograd(cuda_dev):
    import gpytorch_b200 as gp
    from gpytorch_b200 import settings

    n, d = 2500, 4
    x, y = om.synthetic_problem(n, d, 0, torch.float32)
    xd, yd = x.to(cuda_dev), y.to(cuda_dev)
    model, lik = _make_model(gp, xd, yd)
    model.covar_module.base_kernel.lengthscale = 0.7
    model.covar_module.outputscale = 1.4
    lik.noise = 0.2
    mll = gp.mlls.ExactMarginalLogLikelihood(lik, model)
    model.train(); lik.train()
    with settings.max_preconditioner_size(50), settings.cg_tolerance(1e-3), settings.num_trace_samples(16 - 1), settings.probe_seed(3):
        loss = -mll(model(xd), yd)
        loss.backward()
    # dense fp64 autograd reference of the same objective
    ls = torch.tensor(0.7, dtype=torch.float64, requires_grad=True)
    osc = torch.tensor(1.4, dtype=torch.float64, requires_grad=True)
    nz = torch.tensor(0.2, dtype=torch.float64, requires_grad=True)
    K = ok.kernel_matrix("rbf", x.double(), x.double(), ls, osc, True) + nz * torch.eye(n, dtype=torch.float64)
    Lc = torch.linalg.cholesky(K)
    r = y.double().unsqueeze(-1)
    ref = 0.5 * ((r * torch.cholesky_solve(r, Lc)).sum() + 2 * Lc.diagonal().log().sum() + n * math.log(2 * math.pi)) / n
    ref.backward()
    assert loss.item() == pytest.approx(ref.item(), rel=2e-2)
    # chain rule through softplus: d raw = d value * sigmoid(raw)
    k = model.covar_module
    g_ls = k.base_kernel.raw_lengthscale.grad.item() / torch.sigmoid(k.base_kernel.raw_lengthscale).item()
    g_os = k.raw_outputscale.grad.item() / torch.sigmoid(k.raw_outputscale).item()
    g_nz = lik.raw_noise.grad.item() / torch.sigmoid(lik.raw_noise).item()
    # stochastic trace estimate with 15 probes: gradients agree to ~10 %
    assert g_ls == pytest.approx(ls.grad.item(), rel=0.15, abs=2e-3)
    assert g_os == pytest.approx(osc.grad.item(), rel=0.15, abs=2e-3)
    assert g_nz == pytest.approx(nz.grad.item(), rel=0.15, abs=2e-3)


def test_api_small_n_uses_cholesky_branch_and_matches_exactly(cuda_dev):
    import gpytorch_b200 as gp

    n = 300  # <= max_cholesky_size: the reference's dense branch
    x, y = om.synthetic_problem(n, 2, 0, torch.float32)
    model, lik = _make_model(gp, x.to(cuda_dev), y.to(cuda_dev), kind="matern52")
    lik.noise = 0.1
    mll = gp.mlls.ExactMarginalLogLikelihood(lik, model)
    model.train()
    out = mll(model(x.to(cuda_dev)), y.to(cuda_dev))
    ls = model.covar_module.base_kernel.lengthscale.item(); osc = model.covar_module.outputscale.item()
    ch = om.mll_cholesky("matern52", x.double(), y.double(), 0.0, ls, osc, 0.1)
    assert out.item() == pytest.approx(ch.mll, rel=1e-3)


def test_api_training_reduces_loss_and_prediction_mae(cuda_dev):
    # end-to-end on the CG path, like /root/reference/test/examples/test_white_noise_regression.py:57-102 (max_cholesky_size(0))
    import gpytorch_b200 as gp
    from gpytorch_b200 import settings

    g = torch.Generator().manual_seed(0)
    train_x = torch.linspace(0, 1, 900).unsqueeze(-1)
    train_y = torch.sin(train_x[:, 0] * 2 * math.pi) + 0.05 * torch.randn(900, generator=g)
    test_x = torch.linspace(0.02, 0.98, 51).unsqueeze(-1)
    test_y = torch.sin(test_x[:, 0] * 2 * math.pi)
    xd, yd = train_x.to(cuda_dev), train_y.to(cuda_dev)
    model, lik = _make_model(gp, xd, yd)
    mll = gp.mlls.ExactMarginalLogLikelihood(lik, model)
    opt = torch.optim.Adam(model.parameters(), lr=0.1)
    model.train(); lik.train()
    losses = []
    with settings.max_cholesky_size(0), settings.min_preconditioning_size(100), settings.cg_tolerance(0.05), settings.probe_seed(0):
        for _ in range(30):
            opt.zero_grad()
            loss = -mll(model(xd), yd)
            loss.backward()
            opt.step()
            losses.append(loss.item())
        model.eval(); lik.eval()
        with torch.no_grad():
            pred = model(test_x.to(cuda_dev))
    assert losses[-1] < losses[0] - 0.3
    mae = (pred.mean.cpu() - test_y).abs().mean().item()
    assert mae < 0.05
    assert torch.all(pred.variance > -1e-3)


def test_api_function_seam_linear_cg_signature(cuda_dev):
    import gpytorch_b200 as gp

    n = 1200
    x, y = om.synthetic_problem(n, 3, 0, torch.float32)
    op = gp.kernels.ScaleKernel(gp.kernels.RBFKernel()).to(cuda_dev)(x.to(cuda_dev))
    khat = op.add_jitter(0.5)
    rhs = torch.randn(n, 3).to(cuda_dev)
    sol = gp.linear_cg(khat.matmul, rhs, n_tridiag=0, tolerance=1e-4, max_iter=500, max_tridiag_iter=10)
    assert rel(khat.matmul(sol), rhs) < 1e-3
    sol2, tmat = gp.linear_cg(khat.matmul, rhs, n_tridiag=2, tolerance=1e-4, max_iter=500, max_tridiag_iter=10)
    assert tmat.shape[0] == 2 and tmat.shape[-1] == tmat.shape[-2] <= 10
    L = gp.pivoted_cholesky(op, 20)
    assert L.shape == (n, 20)


def test_api_love_fast_pred_var_matches_oracle_and_exact(cuda_dev):
    """SURVEY 8(f) row 2: LOVE predictive covariance (settings.fast_pred_var; exact_prediction_strategies.py:268-272,
    464-478) on the engine's Lanczos + fused cross-covariance K.V, against the oracle's restatement with the same
    start vector (fp64) and against the exact predictive covariance."""
    import gpytorch_b200 as gp
    from gpytorch_b200 import settings
    from oracle import linalg as ol

    n, m, d = 2600, 40, 3
    x, y = om.synthetic_problem(n, d, 0, torch.float32)
    g = torch.Generator().manual_seed(5)
    xs = torch.rand(m, d, generator=g)
    model, lik = _make_model(gp, x.to(cuda_dev), y.to(cuda_dev))
    model.covar_module.base_kernel.lengthscale = 0.6
    model.covar_module.outputscale = 1.3
    lik.noise = 0.15
    model.eval(); lik.eval()
    with torch.no_grad(), settings.probe_seed(7), settings.max_root_decomposition_size(60), settings.eval_cg_tolerance(1e-4):
        with settings.fast_pred_var(True):
            love = model(xs.to(cuda_dev)).covariance_matrix.cpu().double()
        exact = model(xs.to(cuda_dev)).covariance_matrix.cpu().double()
        with settings.skip_posterior_variances(True):
            assert float(model(xs.to(cuda_dev)).covariance_matrix.abs().max()) == 0.0
    # oracle, fp64, same start vector
    xd, xsd = x.double(), xs.double()
    K = ok.kernel_matrix("rbf", xd, xd, 0.6, 1.3, True) + 0.15 * torch.eye(n, dtype=torch.float64)
    ksx = ok.kernel_matrix("rbf", xsd, xd, 0.6, 1.3, False)
    kss = ok.kernel_matrix("rbf", xsd, xsd, 0.6, 1.3, True)
    init = torch.randn(n, generator=torch.Generator().manual_seed(7)).double()
    r = ol.root_inv_decomposition(lambda v: K @ v, 60, init)
    o_love = ol.love_predictive_covar(kss, ksx, r)
    K32 = K.float()
    r32 = ol.root_inv_decomposition(lambda v: K32 @ v, 60, init.float())          # the reference's own default dtype
    o_love32 = ol.love_predictive_covar(kss.float(), ksx.float(), r32).double()
    o_exact = kss - ksx @ torch.linalg.solve(K, ksx.T)
    scale = o_exact.diagonal().mean().item()
    # the truncated Krylov inverse amplifies fp32 rounding by cond(K_hat) ~ 1e4: stated tolerance = 2e-3 of the mean
    # predictive variance, or no further from the fp64 oracle than 3x the fp32 run of the same algorithm
    dev32 = (o_love32 - o_love).abs().max().item()
    assert (love - o_love).abs().max().item() <= max(2e-3 * scale, 3 * dev32), ((love - o_love).abs().max().item(), dev32, scale)
    # K** - K*x K_hat^-1 Kx* cancels from ~1.3 to ~2e-3: the CG solve (eval_cg_tolerance 1e-4, fp32) leaves an absolute
    # error of ~tol * outputscale in every entry (the reference's default eval tolerance is 1e-2)
    assert (exact - o_exact).abs().max().item() < 1e-3 * 1.3
    # LOVE itself is an approximation of the exact covariance (60 Lanczos steps): loose, like the reference's own test
    # (test/examples/test_simple_gp_regression.py: fast_pred_var variances within ~1e-2..5e-2)
    assert (love.diagonal() - exact.diagonal()).abs().max().item() < 5e-2 * scale + 1e-3


def test_api_operator_seam_protocol_and_solve_vs_dense_inverse(cuda_dev):
    """SURVEY 8(b) operator seam: the LinearOperator subset the reference's callers use, and the reference's own
    solve-through-CG check (test/lazy/test_lazy_evaluated_kernel_tensor.py:69-113: vs evaluated.inverse(), rtol 0.02 /
    atol 1e-5 under cg_tolerance(1e-4), gradients wrt the kernel parameters and the right-hand side)."""
    import gpytorch_b200 as gp
    from gpytorch_b200 import settings

    n, m, d = 1100, 300, 3
    x, _ = om.synthetic_problem(n, d, 0, torch.float32)
    x2 = torch.rand(m, d, generator=torch.Generator().manual_seed(9))
    kern = gp.kernels.ScaleKernel(gp.kernels.RBFKernel()).to(cuda_dev)
    kern.base_kernel.lengthscale = 0.6
    kern.outputscale = 1.2
    op = kern(x.to(cuda_dev))
    cross = kern(x.to(cuda_dev), x2.to(cuda_dev))
    Kd = ok.kernel_matrix("rbf", x.double(), x.double(), 0.6, 1.2, True)
    Kx = ok.kernel_matrix("rbf", x.double(), x2.double(), 0.6, 1.2, False)
    # shape protocol
    assert op.shape == op._size() == op.matrix_shape == torch.Size([n, n]) and op.dim() == 2 and op.numel() == n * n
    assert cross.shape == torch.Size([n, m]) and cross.t().shape == cross.mT.shape == cross.transpose(-1, -2).shape == torch.Size([m, n])
    assert op.batch_shape == torch.Size([]) and op.dtype == torch.float32 and op.device.type == "cuda" and op.requires_grad
    assert len(op.representation()) == 4 and op.evaluate_kernel() is op and op.t() is op
    # products: matmul / @ / transpose / diagonal / getitem / to_dense
    v = torch.randn(m, 3, generator=torch.Generator().manual_seed(1))
    w = torch.randn(n, 2, generator=torch.Generator().manual_seed(2))
    assert rel((cross @ v.to(cuda_dev)).detach(), Kx @ v.double()) < 5e-6
    assert rel(cross.t().matmul(w.to(cuda_dev)).detach(), Kx.T @ w.double()) < 5e-6
    assert rel(op.diagonal().detach(), Kd.diagonal()) < 1e-6 and rel(op._diagonal().detach(), Kd.diagonal()) < 1e-6
    assert rel(op[5:40, 100:260].to_dense().detach(), Kd[5:40, 100:260]) < 5e-6
    assert rel(op._getitem(slice(0, 16), slice(None)).to_dense().detach(), Kd[:16]) < 5e-6
    khat = op + gp.operators.ConstantDiagLinearOperator(torch.tensor(0.3, device=cuda_dev), n)
    khat2 = khat.add_jitter(0.2)
    assert float(khat2.noise) == pytest.approx(0.5) and khat.t() is khat and khat.shape == op.shape and khat.requires_grad
    assert rel(khat2.diagonal().detach(), Kd.diagonal() + 0.5) < 1e-6
    assert rel((khat @ w.to(cuda_dev)).detach(), (Kd + 0.3 * torch.eye(n, dtype=torch.float64)) @ w.double()) < 5e-6
    # solve through CG vs the dense inverse, with gradients (the reference's _test_inv_matmul)
    rhs = torch.randn(n, 4, generator=torch.Generator().manual_seed(3)).to(cuda_dev).requires_grad_(True)
    with settings.max_cholesky_size(0), settings.cg_tolerance(1e-4), settings.max_preconditioner_size(30):
        res = khat.solve(rhs)
        grad = torch.randn(n, 4, generator=torch.Generator().manual_seed(4))
        res.backward(gradient=grad.to(cuda_dev))
    ls = torch.tensor(0.6, dtype=torch.float64, requires_grad=True)
    osc = torch.tensor(1.2, dtype=torch.float64, requires_grad=True)
    rhs_c = rhs.detach().cpu().double().requires_grad_(True)
    Ka = ok.kernel_matrix("rbf", x.double(), x.double(), ls, osc, True) + 0.3 * torch.eye(n, dtype=torch.float64)
    actual = torch.linalg.solve(Ka, rhs_c)
    actual.backward(gradient=grad.double())
    # the reference's own bound is rtol 0.02 / atol 1e-5 on a 5 x 5 system; at n = 1100 with cg_tolerance(1e-4) the fp32
    # solve carries ~1e-4 of the solution norm in every entry, so the absolute part is scaled accordingly
    assert rel(res.detach(), actual.detach()) < 1e-3
    assert torch.allclose(res.detach().cpu().double(), actual.detach(), rtol=0.02, atol=2e-3)
    g_ls = kern.base_kernel.raw_lengthscale.grad.item() / torch.sigmoid(kern.base_kernel.raw_lengthscale).item()
    g_os = kern.raw_outputscale.grad.item() / torch.sigmoid(kern.raw_outputscale).item()
    assert g_ls == pytest.approx(ls.grad.item(), rel=1e-2, abs=1e-3)
    assert g_os == pytest.approx(osc.grad.item(), rel=1e-2, abs=1e-3)
    assert rel(rhs.grad, rhs_c.grad) < 1e-3 and torch.allclose(rhs.grad.cpu().double(), rhs_c.grad, rtol=0.03, atol=2e-3)
    # log-det / inv-quad shortcuts
    with settings.max_cholesky_size(0), settings.probe_seed(0), settings.num_trace_samples(15), settings.max_preconditioner_size(30):
        ld = khat.logdet().item()
        iq = khat.inv_quad(rhs.detach()[:, :1]).item()
    assert ld == pytest.approx(torch.logdet(Ka.detach()).item(), rel=5e-2)
    assert iq == pytest.approx((rhs_c.detach()[:, :1] * torch.linalg.solve(Ka.detach(), rhs_c.detach()[:, :1])).sum().item(), rel=1e-3)
