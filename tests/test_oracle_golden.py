"""Pins the oracle: CPU restatement vs outputs of the reference's own code (tests/golden/kernels_golden.npz,
made by tests/golden/make_golden.py) and vs the known answers in the reference's tests."""
import math

import numpy as np
import pytest
import torch

from oracle import kernels as ok, linalg as ol, mll as om

CASES = ["a", "b", "c", "d"]


@pytest.mark.parametrize("tag", CASES)
@pytest.mark.parametrize("dt", ["f32", "f64"])
def test_kernels_match_reference_outputs(golden, tag, dt):
    key = f"{tag}_{dt}"
    x1 = torch.from_numpy(golden[f"{key}_x1"])
    same = bool(golden[f"{key}_same"])
    x2 = x1 if same else torch.from_numpy(golden[f"{key}_x2"])
    ls = float(golden[f"{key}_ls"])
    rows = golden[f"{key}_rows"]  # the golden file holds these rows of each reference matrix
    tol = dict(rtol=1e-5, atol=1e-6) if dt == "f32" else dict(rtol=1e-12, atol=1e-13)
    np.testing.assert_allclose(ok.sq_dist(x1, x2, same).numpy()[rows], golden[f"{key}_sqdist"], **tol)
    np.testing.assert_allclose(ok.dist(x1, x2, same).numpy()[rows], golden[f"{key}_dist"], **tol)
    np.testing.assert_allclose(ok.rbf(x1, x2, ls, same).numpy()[rows], golden[f"{key}_rbf"], **tol)
    for nu, nk in ((0.5, "mat12"), (1.5, "mat32"), (2.5, "mat52")):
        np.testing.assert_allclose(ok.matern(x1, x2, ls, nu, same).numpy()[rows], golden[f"{key}_{nk}"], **tol)
    lsv = torch.from_numpy(golden[f"{key}_ard_ls"])
    np.testing.assert_allclose(ok.rbf(x1, x2, lsv, same).numpy()[rows], golden[f"{key}_rbf_ard"], **tol)


@pytest.mark.parametrize("tag", CASES)
def test_lengthscale_gradient_matches_reference_autograd(golden, tag):
    key = f"{tag}_f64"
    x1 = torch.from_numpy(golden[f"{key}_x1"])
    same = bool(golden[f"{key}_same"])
    x2 = x1 if same else torch.from_numpy(golden[f"{key}_x2"])
    ls = float(golden[f"{key}_ls"])
    W = torch.outer(torch.from_numpy(golden[f"{key}_w_u"]), torch.from_numpy(golden[f"{key}_w_v"]))
    for kind, nk in (("rbf", "rbf"), ("matern12", "mat12"), ("matern32", "mat32"), ("matern52", "mat52")):
        g = (ok.dk_dlengthscale(kind, x1, x2, ls, same) * W).sum().item()
        assert g == pytest.approx(float(golden[f"{key}_{nk}_dls"].reshape(-1)[0]), rel=1e-9)


def test_rbf_known_answer():
    # /root/reference/test/kernels/test_rbf_kernel.py:126-137
    a = torch.tensor([4.0, 2.0, 8.0]).view(3, 1)
    b = torch.tensor([0.0, 2.0, 4.0]).view(3, 1)
    actual = torch.tensor([[16.0, 4, 0], [4, 0, 4], [64, 36, 16]]).mul_(-0.5).div_(4.0).exp_()
    assert torch.norm(ok.rbf(a, b, 2.0) - actual) < 1e-5


def test_matern_known_answers():
    # /root/reference/test/kernels/test_matern_kernel.py:41-75
    a = torch.tensor([4.0, 2.0, 8.0]).view(3, 1)
    b = torch.tensor([0.0, 2.0]).view(2, 1)
    d = torch.tensor([[4.0, 2], [2, 0], [8, 6]])
    assert torch.norm(ok.matern(a, b, 2.0, 0.5) - d.div(-2.0).exp()) < 1e-3
    r = d * math.sqrt(3) / 2
    assert torch.norm(ok.matern(a, b, 2.0, 1.5) - (r + 1) * torch.exp(-r)) < 1e-3
    r = d * math.sqrt(5) / 2
    assert torch.norm(ok.matern(a, b, 2.0, 2.5) - (r**2 / 3 + r + 1) * torch.exp(-r)) < 1e-3


def test_matern_ard_known_answer():
    # /root/reference/test/kernels/test_matern_kernel.py:77-90
    a = torch.tensor([[1.0, 2], [3, 4]])
    b = torch.tensor([[1.0, 4], [1, 4]])
    dist = torch.tensor([[1.0, 1], [2, 2]]) * math.sqrt(5)
    actual = (dist**2 / 3 + dist + 1) * torch.exp(-dist)
    assert torch.norm(ok.matern(a, b, torch.tensor([1.0, 2.0]), 2.5) - actual) < 1e-3


def test_scale_kernel():
    # outputscale multiplies K (kernels/scale_kernel.py:108-118; test/kernels/test_scale_kernel.py:24-58)
    x = torch.rand(7, 2, dtype=torch.float64)
    assert torch.allclose(ok.kernel_matrix("rbf", x, x, 0.7, 3.0), 3.0 * ok.rbf(x, x, 0.7))


def test_log_prob_known_answer():
    # /root/reference/test/distributions/test_multivariate_normal.py:23-43: log_prob(0) = -4.8157
    mean = torch.tensor([0.0, 1, 2], dtype=torch.float64)
    var = torch.tensor([1.0, 0.75, 1.5], dtype=torch.float64)
    diff = -mean
    inv_quad = (diff**2 / var).sum()
    logdet = var.log().sum()
    lp = -0.5 * (inv_quad + logdet + 3 * math.log(2 * math.pi))
    assert lp.item() == pytest.approx(-4.8157, abs=1e-4)


# ---- linear-algebra half: no reference golden exists ("parity unpinned"); anchored on dense ground truth ----
@pytest.fixture(scope="module")
def problem():
    n, d = 600, 3
    x, y = om.synthetic_problem(n, d, 0, torch.float64)
    K = ok.kernel_matrix("rbf", x, x, 0.5, 1.0, True)
    return n, x, y, K, K + 0.1 * torch.eye(n, dtype=torch.float64)


def test_linear_cg_converges_to_dense_solve(problem):
    n, x, y, K, A = problem
    rhs = torch.randn(n, 4, dtype=torch.float64, generator=torch.Generator().manual_seed(1))
    # the eps=1e-10 guards on p^T A p make the recurrence stall near |r| ~ 1e-6 (reference behaviour), so ask for 1e-5
    sol = ol.linear_cg(lambda v: A @ v, rhs, tolerance=1e-5, max_iter=2000)
    ref = torch.linalg.solve(A, rhs)
    assert (sol - ref).norm() / ref.norm() < 1e-4


def test_linear_cg_default_iteration_count_and_tridiag_shape(problem):
    n, x, y, K, A = problem
    rhs = torch.randn(n, 11, dtype=torch.float64, generator=torch.Generator().manual_seed(2))
    with _nullctx():
        sol, tmat, info = ol.linear_cg(lambda v: A @ v, rhs, n_tridiag=10, return_info=True)
    assert info.iters == 21  # SURVEY.md Appendix A.2: 20 tridiag iterations are forced, stop at k = 20
    assert tmat.shape == (10, 20, 20)
    assert torch.allclose(tmat, tmat.transpose(-1, -2))


class _nullctx:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def test_cg_tridiag_matches_lanczos_spectrum(problem):
    # the CG-derived tridiagonal is the Lanczos tridiagonal of A started at rhs/|rhs|
    n, x, y, K, A = problem
    rhs = torch.randn(n, 1, dtype=torch.float64, generator=torch.Generator().manual_seed(3))
    _, tmat = ol.linear_cg(lambda v: A @ v, rhs, n_tridiag=1, max_tridiag_iter=12, tolerance=1e-12, max_iter=400)
    _, T = ol.lanczos_tridiag(lambda v: A @ v, 12, rhs)
    assert torch.allclose(torch.linalg.eigvalsh(tmat[0]), torch.linalg.eigvalsh(T[0]), rtol=1e-4, atol=1e-6)


def test_pivoted_cholesky_and_preconditioner(problem):
    n, x, y, K, A = problem
    L, piv = ol.pivoted_cholesky(K.diagonal().clone(), lambda i: K[i], 40, 1e-12)
    assert L.shape == (n, 40) and len(set(piv.tolist())) == 40
    # exact on the pivot rows, residual diagonal non-negative and trace decreasing
    R = K - L @ L.t()
    assert R[piv].abs().max() < 1e-8
    assert R.diagonal().min() > -1e-10
    L20, _ = ol.pivoted_cholesky(K.diagonal().clone(), lambda i: K[i], 20, 1e-12)
    assert (K - L20 @ L20.t()).diagonal().sum() > R.diagonal().sum()
    pre = ol.build_preconditioner(L, 0.1)
    P = L @ L.t() + 0.1 * torch.eye(n, dtype=torch.float64)
    v = torch.randn(n, 3, dtype=torch.float64)
    assert torch.allclose(pre.apply(v), torch.linalg.solve(P, v), rtol=1e-8, atol=1e-9)
    assert pre.logdet == pytest.approx(torch.logdet(P).item(), rel=1e-10)


def test_pivoted_cholesky_stops_on_tolerance(problem):
    n, x, y, K, A = problem
    L, piv = ol.pivoted_cholesky(K.diagonal().clone(), lambda i: K[i], 500, 1e-1)
    assert L.size(1) < 500
    resid = (K - L @ L.t()).diagonal()
    mask = torch.ones(n, dtype=torch.bool); mask[piv] = False
    assert resid[mask].abs().sum() / 1.0 <= 1e-1


def test_mll_bbmm_close_to_cholesky():
    n, d = 1000, 3
    x, y = om.synthetic_problem(n, d, 0, torch.float64)
    pn = tuple(a.double() for a in om.make_probe_noise(n, 15, 10, 1))
    ch = om.mll_cholesky("rbf", x, y, 0.0, 0.5, 1.0, 0.1)
    r = om.mll_bbmm("rbf", x, y, 0.0, 0.5, 1.0, 0.1, pn, min_precond_size=0)
    assert r.iters == 21
    assert r.inv_quad == pytest.approx(ch.inv_quad, rel=1e-6)      # SURVEY.md Appendix A: 147.14992 both
    assert r.logdet == pytest.approx(ch.logdet, rel=2e-2)          # 10 probes: statistical agreement
    r0 = om.mll_bbmm("rbf", x, y, 0.0, 0.5, 1.0, 0.1, pn)          # n < 2000: no preconditioner, Rademacher probes
    assert r0.precond is None and r0.inv_quad == pytest.approx(ch.inv_quad, rel=5e-3)


def test_lanczos_orthogonal_basis(problem):
    n, x, y, K, A = problem
    Q, T = ol.lanczos_tridiag(lambda v: A @ v, 25, torch.randn(n, 1, dtype=torch.float64))
    Q, T = Q[0], T[0]
    assert (Q.t() @ Q - torch.eye(T.size(0), dtype=torch.float64)).abs().max() < 1e-10
    assert (Q.t() @ A @ Q - T).abs().max() < 1e-8


def test_per_row_noise_preconditioner_and_mll_against_dense():
    """Groundwork for FixedNoiseGaussianLikelihood (likelihoods/gaussian_likelihood.py:245-363, SURVEY 8f row 4): the
    non-constant-diagonal preconditioner branch and the BBMM MLL with a per-row noise vector vs dense linear algebra."""
    torch.manual_seed(3)
    n, k = 400, 12
    x, y = om.synthetic_problem(n, 3, 0, torch.float64)
    K = ok.kernel_matrix("rbf", x, x, 0.6, 1.0, True)
    d = 0.05 + 0.3 * torch.rand(n, dtype=torch.float64)
    L, piv = ol.pivoted_cholesky(torch.ones(n, dtype=torch.float64), lambda i: K[i], k, 1e-6)
    pre = ol.build_preconditioner(L, d, piv)
    P = L @ L.t() + torch.diag(d)
    v = torch.randn(n, 3, dtype=torch.float64)
    assert (pre.apply(v) - torch.linalg.solve(P, v)).abs().max().item() < 1e-9
    assert pre.logdet == pytest.approx(torch.logdet(P).item(), rel=1e-10)
    e1, e2 = torch.randn(L.size(1), 20000, dtype=torch.float64), torch.randn(n, 20000, dtype=torch.float64)
    z = pre.probes(e1, e2)
    emp = (z[:5] @ z[:5].t()) / 20000
    assert (emp - P[:5, :5]).abs().max().item() < 0.06           # z ~ N(0, P)
    # constant vector == scalar branch
    pre_c = ol.build_preconditioner(L, torch.full((n,), 0.2, dtype=torch.float64), piv)
    pre_s = ol.build_preconditioner(L, 0.2, piv)
    assert (pre_c.apply(v) - pre_s.apply(v)).abs().max().item() < 1e-10 and pre_c.logdet == pytest.approx(pre_s.logdet, rel=1e-12)
    # MLL with per-row noise: mBCG/SLQ vs dense Cholesky
    n2 = 2100
    x2, y2 = om.synthetic_problem(n2, 3, 0, torch.float64)
    d2 = 0.05 + 0.2 * torch.rand(n2, dtype=torch.float64)
    pn = tuple(a.double() for a in om.make_probe_noise(n2, 30, 10, 1))
    ch = om.mll_cholesky("rbf", x2, y2, 0.0, 0.7, 1.0, d2)
    bb = om.mll_bbmm("rbf", x2, y2, 0.0, 0.7, 1.0, d2, pn, precond_size=30, tolerance=1e-3)
    assert bb.inv_quad == pytest.approx(ch.inv_quad, rel=1e-3)
    assert bb.logdet == pytest.approx(ch.logdet, rel=3e-2)
