#!/usr/bin/env python
"""Linearised and Laplace uncertainties of the test_1 model (raytracerfortran_b200.grad).

Starts from the test_1 MAP model with its data and sigma.  That model is not a minimum of the
misfit (1/2) |tobs - T|^2 (there the exact Newton matrix has a negative eigenvalue), so the example
first refines it by Levenberg-Marquardt on the Gauss-Newton normal equations.  At the refined
model it prints the 1-sigma value of every parameter from the Gauss-Newton covariance
(J^T J / sigma^2)^-1 next to the one from the Laplace (Gaussian) approximation of the posterior,
(A / sigma^2)^-1, where A = J^T J - sum_s r_s d2T_s is the exact Newton matrix
(grad.newton_equations).  Their ratio shows how much the residual-weighted second derivatives,
which Gauss-Newton leaves out, move each value.  Parameters reached by fewer than two rays (the
deepest layer and interface, seen by one source) are not determined by the data and are left out
of both matrices.  The library returns the matrices; every solve is done here.  Exits non-zero if
A is not exactly symmetric or the Cholesky factorisation of A / sigma^2 fails.

    python examples/laplace_test1.py
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from raytracerfortran_b200 import grad  # noqa: E402


def main():
    c = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_golden.json")))["config1"]
    dev = torch.device("cuda:0")
    t = lambda a: torch.tensor(np.asarray(a, dtype=np.float64), device=dev)
    v0, z0 = t(c["vels"]), t(c["depths"])
    so, sd, tobs = t(c["src_offset_full"]), t(c["src_depth_full"]), t(c["tobs"])
    nv, nz = v0.numel(), z0.numel()
    nl = torch.tensor([nz], dtype=torch.int32, device=dev)
    sigma = float(c["sigma_map"])

    def newton(x):
        N = grad.newton_equations(x[None, :nv], x[None, nv:], nl, so, sd, tobs)
        r = tobs - N["timeP"][0]
        return N, float((r * r).sum())

    def valid(x):
        z = x[nv:]
        return bool((x[:nv] > 0).all() and z[0] > 0 and (z[1:] > z[:-1]).all())

    # columns reached by at least two rays: a ray reaches velocity i < n and interface j <= n - 2
    n = 1 + (sd[:, None] > z0[None, :]).sum(1)
    rays = torch.cat([(n[:, None] > torch.arange(nv, device=dev)).sum(0),
                      (n[:, None] - 2 >= torch.arange(nz, device=dev)).sum(0)])
    keep = rays >= 2
    k2 = keep[:, None] & keep[None, :]
    m = int(keep.sum())

    # Levenberg-Marquardt on J^T J from the MAP model, damping with diag(J^T J)
    x = torch.cat([v0, z0])
    N, ss = newton(x)
    ss0, lam, it = ss, 1e-3, 0
    for it in range(1, 201):
        G = N["JtJ"][0][k2].view(m, m)
        dx = torch.linalg.solve(G + lam * torch.diag(torch.diagonal(G)), N["Jtr"][0][keep])
        xn = x.clone()
        xn[keep] += dx
        if valid(xn):
            Nn, ssn = newton(xn)
            if ssn < ss:
                done = ss - ssn < 1e-12 * ss
                x, N, ss, lam = xn, Nn, ssn, lam / 3
                if done:
                    break
                continue
        lam *= 4
        if lam > 1e12:
            break

    A = N["A"][0]
    if not torch.equal(A, A.T):
        sys.exit("the Newton matrix is not exactly symmetric")
    L, info = torch.linalg.cholesky_ex(A[k2].view(m, m) / sigma ** 2)
    if int(info) != 0:
        sys.exit(f"the Laplace matrix A / sigma^2 is not positive definite (Cholesky failed at {int(info)})")
    Lg, info_gn = torch.linalg.cholesky_ex(N["JtJ"][0][k2].view(m, m) / sigma ** 2)
    sd_lp = torch.sqrt(torch.diagonal(torch.cholesky_inverse(L)))
    sd_gn = torch.sqrt(torch.diagonal(torch.cholesky_inverse(Lg)))
    if int(info_gn) != 0:
        sd_gn = torch.full_like(sd_gn, float("nan"))
    print(f"test_1: {so.numel()} rays, sigma = {sigma:g} s; sum of squared residuals {ss0:.6g} s^2 at the "
          f"MAP model, {ss:.6g} s^2 after {it} Levenberg-Marquardt iterations")
    print(f"{'parameter':>10} {'MAP':>10} {'refined':>10} {'rays':>5} {'1-sigma GN':>12} {'1-sigma Laplace':>16} "
          f"{'ratio':>7}")
    names = [f"V{i}" for i in range(nv)] + [f"z{j}" for j in range(nz)]
    x0 = torch.cat([v0, z0])
    k = 0
    for i, name in enumerate(names):
        line = f"{name:>10} {float(x0[i]):10.2f} {float(x[i]):10.2f} {int(rays[i]):5d}"
        if keep[i]:
            line += f" {float(sd_gn[k]):12.4g} {float(sd_lp[k]):16.4g} {float(sd_lp[k] / sd_gn[k]):7.4f}"
            k += 1
        else:
            line += f" {'not determined (fewer than two rays)':>37}"
        print(line)


if __name__ == "__main__":
    main()
