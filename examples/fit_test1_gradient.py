#!/usr/bin/env python
"""Fit the test_1 model to its travel times with gradients (raytracerfortran_b200.grad).

Start from a perturbed model (velocities +-10 %, interfaces +-50 m, the number of layers fixed) and
maximise LOGLHOOD_RT with torch.optim.LBFGS, on the GPU.  The fit runs in slowness (s/km) and
interface depth (km): travel times are nearly linear in slowness and both sets of unknowns then
have gradients of similar size (in m/s the low-velocity second layer stalls the search).  The
misfit is not convex, so another seed can end in a local maximum.  Exits non-zero unless the fit
ends no lower than the true model's logL - 1.

    python examples/fit_test1_gradient.py [--seed S]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from raytracerfortran_b200 import grad  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seed", type=int, default=1)
    args = ap.parse_args()
    c = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_golden.json")))["config1"]
    dev = torch.device("cuda:0")
    t = lambda a: torch.tensor(np.asarray(a, dtype=np.float64)[None], device=dev)
    v_true, z_true = t(c["vels"]), t(c["depths"])
    so, sd = t(c["src_offset_full"])[0], t(c["src_depth_full"])[0]
    tobs = t(c["tobs"])[0]
    sigma = torch.tensor([c["sigma_map"]], dtype=torch.float64, device=dev)
    nl = torch.tensor([z_true.shape[1]], dtype=torch.int32, device=dev)

    def logl(v, z):
        return grad.loglhood(v, z, nl, so, sd, tobs, sigma)[0]

    rng = np.random.default_rng(args.seed)
    v0 = v_true * torch.tensor(1.0 + rng.uniform(-0.1, 0.1, v_true.shape), device=dev)
    z0 = z_true + torch.tensor(rng.uniform(-50.0, 50.0, z_true.shape), device=dev)
    xs = (1000.0 / v0).clone().requires_grad_(True)       # slowness, s/km
    xz = (z0 / 1000.0).clone().requires_grad_(True)       # interface depth, km
    opt = torch.optim.LBFGS([xs, xz], lr=1.0, max_iter=200, tolerance_grad=1e-12,
                            tolerance_change=1e-14, history_size=20, line_search_fn="strong_wolfe")

    def closure():
        opt.zero_grad()
        loss = -logl(1000.0 / xs, xz * 1000.0)
        loss.backward()
        return loss

    with torch.no_grad():
        l_true, l_start = logl(v_true, z_true).item(), logl(v0, z0).item()
    for _ in range(5):
        opt.step(closure)
    with torch.no_grad():
        l_fit = logl(1000.0 / xs, xz * 1000.0).item()
    print(f"logL: start {l_start:.3f}, fit {l_fit:.3f}, true model {l_true:.3f}")
    print("velocities (m/s):", np.round((1000.0 / xs).detach().cpu().numpy()[0], 1).tolist())
    print("true:            ", c["vels"])
    print("interfaces (m):  ", np.round((xz * 1000.0).detach().cpu().numpy()[0], 1).tolist())
    print("true:            ", c["depths"])
    if not l_fit >= l_true - 1.0:
        sys.exit("the fit ended below the true model's logL - 1")


if __name__ == "__main__":
    main()
