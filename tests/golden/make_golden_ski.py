#!/usr/bin/env python
"""Golden vectors for the SKI / KISS-GP row (SURVEY.md section 8f row 3), produced by EXECUTING the reference's own
code in the build container.  `gpytorch/utils/grid.py` imports only torch and is loaded by path;
`gpytorch/utils/interpolation.py` imports linear_operator (absent) for two helpers it does not use inside
`Interpolation.interpolate`, so its source is read where it lies, the two import statements are dropped and the rest is
executed with `convert_legacy_grid` taken from the loaded grid module.  Nothing is copied into the repo.
Output: tests/golden/ski_golden.npz (committed).
Re-run:  python tests/golden/make_golden_ski.py <path to the gpytorch source tree>
"""
import importlib.util
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))


def load_reference(ref):
    spec = importlib.util.spec_from_file_location("ref_grid", f"{ref}/gpytorch/utils/grid.py")
    grid = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(grid)
    src = open(f"{ref}/gpytorch/utils/interpolation.py").read()
    keep = [ln for ln in src.splitlines()
            if not ln.startswith("from linear_operator") and not ln.startswith("from .grid")]
    ns = {"convert_legacy_grid": grid.convert_legacy_grid, "__name__": "ref_interpolation"}
    exec(compile("\n".join(keep), f"{ref}/gpytorch/utils/interpolation.py", "exec"), ns)
    return grid, ns["Interpolation"]


def main(ref):
    grid_mod, Interpolation = load_reference(ref)
    out = {}
    cases = [("d1", [20], 37), ("d2", [12, 15], 60), ("d3", [8, 9, 10], 50), ("d3c5", [100, 100, 100], 64)]
    for dt_name, dt in (("f32", torch.float32), ("f64", torch.float64)):
        for tag, sizes, npts in cases:
            d = len(sizes)
            g = torch.Generator().manual_seed(77 + d + npts)
            x = torch.rand(npts, d, generator=g, dtype=torch.float64)
            # exercise both boundary branches: points exactly on / next to the data bounds
            x[0] = 0.0
            x[1] = 1.0
            x[2] = 1e-4
            x[3] = 1.0 - 1e-4
            x = x.to(dt)
            bounds = [(0.0, 1.0)] * d
            grid = grid_mod.create_grid(sizes, bounds, extend=True, dtype=dt)
            idx, val = Interpolation().interpolate(grid, x)
            key = f"{tag}_{dt_name}"
            out[f"{key}_x"] = x.numpy()
            for i, gax in enumerate(grid):
                out[f"{key}_grid{i}"] = gax.numpy()
            out[f"{key}_idx"] = idx.numpy()
            out[f"{key}_val"] = val.numpy()
    # the reference's own multi-dimensional known-answer case (test/utils/test_interpolation.py:26-33)
    x = torch.tensor([[0.25, 0.45, 0.65, 0.85], [0.35, 0.375, 0.4, 0.425], [0.45, 0.5, 0.55, 0.6]]).t().contiguous()
    grid = torch.linspace(0.0, 1.0, 11).unsqueeze(1).repeat(1, 3)
    idx, val = Interpolation().interpolate(grid, x)
    out["ka_x"], out["ka_idx"], out["ka_val"] = x.numpy(), idx.numpy(), val.numpy()
    # grid helpers
    out["choose_grid_size_1000_3"] = np.array(grid_mod.choose_grid_size(torch.zeros(1000, 3)))
    out["choose_grid_size_1e6_3"] = np.array(grid_mod.choose_grid_size(torch.zeros(10 ** 6, 3)))
    gd = grid_mod.create_data_from_grid(grid_mod.create_grid([4, 3], [(0.0, 1.0), (2.0, 3.0)], dtype=torch.float64))
    out["grid_data_4x3"] = gd.numpy()
    np.savez_compressed(os.path.join(HERE, "ski_golden.npz"), **out)
    print("wrote", len(out), "arrays")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
