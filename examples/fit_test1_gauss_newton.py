#!/usr/bin/env python
"""Fit the test_1 model from many starts with Levenberg-Marquardt on the per-model normal equations
(raytracerfortran_b200.grad.normal_equations), in torch on the GPU.

1024 starts are perturbed as in fit_test1_gradient.py (velocities +-10 %, interfaces +-50 m, the
number of layers fixed).  The unknowns are slowness (s/km) and interface depth (km), as there; for
them the library's J^T J and J^T r in V and z become S J^T J S and S J^T r with the diagonal chain
rule S = diag(-V^2 / 1000, 1000).  The Jacobian itself is never stored.  Every start has its
own damping lambda: its step solves (J^T J + lambda D) dx = J^T r with D = diag(J^T J), and it
keeps the step only if its own logL rises (then lambda shrinks, otherwise it grows).  All steps of
an iteration are one torch.linalg.solve on [B, P, P].  Prints the best logL against the true
model's, how many starts end within 1 of it, the iteration count, and the linearised standard
deviations of the best fit from (J^T J / sigma^2)^-1.  Exits non-zero unless the best fit ends no
lower than the true model's logL - 1.

    python examples/fit_test1_gauss_newton.py [--seed S] [--starts B] [--iters N]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from raytracerfortran_b200 import device, grad  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--starts", type=int, default=1024)
    ap.add_argument("--iters", type=int, default=100)
    args = ap.parse_args()
    c = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_golden.json")))["config1"]
    dev = torch.device("cuda:0")
    f64 = torch.float64
    t = lambda a: torch.tensor(np.asarray(a, dtype=np.float64), device=dev)
    v_true, z_true = t(c["vels"])[None], t(c["depths"])[None]
    so, sd, tobs = t(c["src_offset_full"]), t(c["src_depth_full"]), t(c["tobs"])
    B, nv, nz = args.starts, v_true.shape[1], z_true.shape[1]
    nl = torch.full((B,), nz, dtype=torch.int32, device=dev)
    sigma = torch.full((B,), c["sigma_map"], dtype=f64, device=dev)

    def logl(v, z):
        # LOGLHOOD_RT of every start; a model with crossing or negative interfaces is not one
        ok = (z[:, :1] > 0).all(1) & (z[:, 1:] > z[:, :-1]).all(1) & (v > 0).all(1)
        L = device.dff_batch_device(v, z, nl[:v.shape[0]], so, sd, tobs=tobs, sigma=sigma[:v.shape[0]])["logL"]
        return torch.where(ok, L, torch.full_like(L, -torch.inf))

    rng = np.random.default_rng(args.seed)
    v0 = v_true * t(1.0 + rng.uniform(-0.1, 0.1, (B, nv)))
    z0 = z_true + t(rng.uniform(-50.0, 50.0, (B, nz)))
    x = torch.cat([1000.0 / v0, z0 / 1000.0], 1)           # slowness (s/km), interface depth (km)
    P = x.shape[1]
    model = lambda x: (1000.0 / x[:, :nv], (x[:, nv:] * 1000.0).contiguous())

    def normal_equations(x):
        v, z = model(x)
        N = grad.normal_equations(v, z, nl[:v.shape[0]], so, sd, tobs=tobs)
        # dT/ds = dT/dV dV/ds = -dT/dV V^2 / 1000,  dT/dz_km = 1000 dT/dz
        S = torch.cat([-(v * v) / 1000.0, torch.full_like(z, 1000.0)], 1)
        return S[:, :, None] * N["JtJ"] * S[:, None, :], S * N["Jtr"]

    L = logl(*model(x))
    l_start = L.clone()
    lam = torch.full((B,), 1e-2, dtype=f64, device=dev)
    eye = torch.eye(P, dtype=f64, device=dev)
    it, quiet = 0, 0
    for it in range(1, args.iters + 1):
        A, g = normal_equations(x)
        D = torch.diagonal(A, dim1=1, dim2=2)
        D = torch.maximum(D, 1e-12 * D.amax(1, keepdim=True))
        dx = torch.linalg.solve(A + lam[:, None, None] * D[:, :, None] * eye, g[:, :, None])[:, :, 0]
        L_new = logl(*model(x + dx))
        acc = L_new > L
        gain = torch.where(acc, L_new - L, torch.zeros_like(L))
        x = torch.where(acc[:, None], x + dx, x)
        L = torch.where(acc, L_new, L)
        lam = torch.where(acc, (lam / 3.0).clamp_min(1e-9), (lam * 3.0).clamp_max(1e12))
        quiet = quiet + 1 if gain.max().item() < 1e-9 else 0
        if quiet >= 5:
            break

    l_true = logl(v_true, z_true)[0].item()
    best = int(torch.argmax(L).item())
    within = int((L >= l_true - 1.0).sum().item())
    print(f"{B} starts, {it} iterations: best logL {L[best].item():.4f}, true model {l_true:.4f}, "
          f"median start {l_start.median().item():.3f}")
    print(f"starts ending within 1 of the true model's logL: {within} of {B}")
    vb, zb = model(x[best:best + 1])
    A, _ = normal_equations(x[best:best + 1])
    cov = torch.linalg.inv(A[0] / (sigma[0] * sigma[0]))
    sd_x = torch.sqrt(torch.diagonal(cov))
    sd_v = sd_x[:nv] * (vb[0] * vb[0]) / 1000.0             # |dV/ds| = V^2 / 1000
    sd_z = sd_x[nv:] * 1000.0
    print("velocities (m/s):   ", np.round(vb[0].cpu().numpy(), 1).tolist())
    print("  1-sigma:          ", np.round(sd_v.cpu().numpy(), 1).tolist())
    print("  true:             ", c["vels"])
    print("interfaces (m):     ", np.round(zb[0].cpu().numpy(), 1).tolist())
    print("  1-sigma:          ", np.round(sd_z.cpu().numpy(), 1).tolist())
    print("  true:             ", c["depths"])
    if not L[best].item() >= l_true - 1.0:
        sys.exit("the best fit ended below the true model's logL - 1")


if __name__ == "__main__":
    main()
