#!/usr/bin/env python
"""Generate golden vectors by EXECUTING the reference's own code (gpytorch source tree, not installed).

`import gpytorch` fails without linear_operator (SURVEY.md section 0), so this
script loads exactly the hot-path pieces that are importable / executable standalone:

* gpytorch/functions/rbf_covariance.py, matern_covariance.py  -> loaded by file path
  (they import only torch/math);
* the bodies of `sq_dist` and `dist` from gpytorch/kernels/kernel.py:26-60 -> extracted
  with `ast` and compiled as-is (the module itself imports linear_operator at the top).

Nothing is copied into the repo: the reference source is read and executed where it lies.
The inputs are stored in full; of every output matrix only the rows `<case>_rows` (a fixed
sample including the first and last row) are stored, and the lengthscale gradients weight K by
the rank-1 matrix W = outer(`<case>_w_u`, `<case>_w_v`), which keeps the file small.
Outputs: tests/golden/kernels_golden.npz (committed).
Re-run:  python tests/golden/make_golden.py <path to the gpytorch source tree>
"""
import ast
import importlib.util
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
N_ROWS = 16


def load_by_path(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def extract_functions(path, names):
    src = open(path).read()
    tree = ast.parse(src)
    ns = {"torch": torch}
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and node.name in names:
            code = compile(ast.Module(body=[node], type_ignores=[]), path, "exec")
            exec(code, ns)
    return [ns[n] for n in names]


def sample_rows(n, seed):
    rest = np.random.default_rng(seed).choice(np.arange(1, n - 1), N_ROWS - 2, replace=False)
    return np.sort(np.concatenate([[0, n - 1], rest])).astype(np.int64)


def main(ref):
    rbf_mod = load_by_path("ref_rbf_cov", f"{ref}/gpytorch/functions/rbf_covariance.py")
    mat_mod = load_by_path("ref_mat_cov", f"{ref}/gpytorch/functions/matern_covariance.py")
    sq_dist, dist = extract_functions(f"{ref}/gpytorch/kernels/kernel.py", ["sq_dist", "dist"])

    out = {}
    cases = [("a", 96, 96, 3, 0.7, True), ("b", 128, 128, 10, 1.3, True), ("c", 70, 45, 10, 0.9, False),
             ("d", 64, 64, 20, 2.0, True)]
    for dt_name, dt in (("f32", torch.float32), ("f64", torch.float64)):
        for tag, n1, n2, d, ls, same in cases:
            g = torch.Generator().manual_seed(1234 + n1 + d)
            x1 = torch.rand(n1, d, generator=g, dtype=torch.float64).to(dt)
            x2 = x1 if same else torch.rand(n2, d, generator=g, dtype=torch.float64).to(dt)
            key = f"{tag}_{dt_name}"
            rows = sample_rows(n1, n1 + d)
            out[f"{key}_rows"] = rows
            out[f"{key}_x1"] = x1.numpy()
            if not same:
                out[f"{key}_x2"] = x2.numpy()
            out[f"{key}_ls"] = np.float64(ls)
            out[f"{key}_same"] = np.bool_(same)
            out[f"{key}_sqdist"] = sq_dist(x1, x2, x1_eq_x2=same).numpy()[rows]
            out[f"{key}_dist"] = dist(x1, x2, x1_eq_x2=same).numpy()[rows]
            # forward + d/dlengthscale through the reference autograd Functions (gradients: fp64 only)
            lsp = torch.tensor([[ls]], dtype=dt, requires_grad=True)
            K = rbf_mod.RBFCovariance.apply(x1, x2, lsp, lambda a, b: sq_dist(a, b, x1_eq_x2=same))
            out[f"{key}_rbf"] = K.detach().numpy()[rows]
            u = torch.rand(n1, generator=g, dtype=torch.float64).to(dt)
            v = torch.rand(n2, generator=g, dtype=torch.float64).to(dt)
            W = torch.outer(u, v)
            grads = dt == torch.float64
            if grads:
                (gl,) = torch.autograd.grad((K * W).sum(), lsp)
                out[f"{key}_w_u"] = u.numpy()
                out[f"{key}_w_v"] = v.numpy()
                out[f"{key}_rbf_dls"] = gl.numpy()
            for nu in (0.5, 1.5, 2.5):
                lsp = torch.tensor([[ls]], dtype=dt, requires_grad=True)
                K = mat_mod.MaternCovariance.apply(x1, x2, lsp, nu, lambda a, b: dist(a, b, x1_eq_x2=same))
                nk = {0.5: "mat12", 1.5: "mat32", 2.5: "mat52"}[nu]
                out[f"{key}_{nk}"] = K.detach().numpy()[rows]
                if grads:
                    (gl,) = torch.autograd.grad((K * W).sum(), lsp)
                    out[f"{key}_{nk}_dls"] = gl.numpy()
            # ARD slow branch of RBFKernel.forward (kernels/rbf_kernel.py:77-79): exp(-0.5 sq_dist(x/l, x/l))
            lsv = torch.linspace(0.5, 1.5, d, dtype=dt)
            out[f"{key}_ard_ls"] = lsv.numpy()
            out[f"{key}_rbf_ard"] = sq_dist(x1 / lsv, x2 / lsv, x1_eq_x2=same).div(-2).exp().numpy()[rows]
    path = os.path.join(HERE, "kernels_golden.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes;", len(out), "arrays")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
