"""numpy restatement of the reverse mode of linear buckling, ``tb_buckling_adjoint`` (TEST INFRASTRUCTURE ONLY).

``factor_grad`` gives the gradients of L = sum_q g_q lambda_q for given critical load factors and K-normalised buckling
modes (the oracle's from ``buckling.buckling`` or the device's), with the member forces N held fixed, and the gradient
with respect to N itself:

  dlambda/dp = lambda phi^T (dK/dp) phi + lambda^2 phi^T (dK_G/dp) phi

per member, with the member geometry of ``oracle/truss_oracle.py`` and the geometric stiffness of ``oracle/buckling.py``.
Composed with ``oracle/adjoint.py`` (g_axial := dL/dN) it gives the total derivative through the static solve.  It is
checked against finite differences of ``buckling.buckling`` and closed forms (tests/test_buckling_adjoint_cpu.py); the
CUDA kernel k_buckling_sens is checked against it (tests/test_gpu_buckling_adjoint.py).
"""
from __future__ import annotations

import numpy as np

from oracle import truss_oracle as orc


def factor_grad(dim, joints, support, conn, aed, axial, factor, modes, g_factor):
    """Gradients of L = sum_q g_factor[q] factor[q] for K-normalised buckling modes (``modes`` [k, N], dense; entries
    at supported DOFs are ignored).  Returns (g_xyz [nJ, d], g_aed [M, 3], g_axial [M]); N is held fixed in g_xyz and
    g_aed.

    Member m from j0 to j1: d = x_j1 - x_j0, L = |d|, c = d / L, k_m = E a / L, g_m = N_m / L, dphi = phi_j1 - phi_j0,
    t = c.dphi, s = |dphi|^2 (phi^T K_m phi = k_m t^2, phi^T K_G,m phi = g_m (s - t^2)):
      dlambda/da = lambda (E/L) t^2,  dlambda/dE = lambda (a/L) t^2,  dlambda/drho = 0,
      dlambda/dN_m = lambda^2 (s - t^2) / L,
      dlambda/dx_j1 = -dlambda/dx_j0 = lambda (k_m/L) (2 t dphi - 3 t^2 c) + lambda^2 (g_m/L) (3 t^2 c - 2 t dphi - s c).
    A mode with g_factor[q] == 0 or a factor that is not finite (+inf: not critical) is skipped.  Exact for simple
    factors; for a cluster only with a cotangent equal across it."""
    joints = np.asarray(joints, dtype=np.float64).reshape(-1, dim)
    conn = np.asarray(conn).astype(np.int64).reshape(-1, 2)
    aed = np.asarray(aed, dtype=np.float64).reshape(-1, 3)
    N_m = np.asarray(axial, dtype=np.float64).reshape(-1)
    nJ = joints.shape[0]
    mask = orc.free_mask(dim, np.asarray(support))
    lam = np.asarray(factor, dtype=np.float64).reshape(-1)
    g = np.asarray(g_factor, dtype=np.float64).reshape(-1)
    use = (g != 0.0) & np.isfinite(lam)
    lam, g = lam[use], g[use]
    phi = np.asarray(modes, dtype=np.float64).reshape(len(use), -1)[use]
    phi = np.where(mask, phi, 0.0).reshape(len(lam), nJ, dim)
    j0, j1 = conn[:, 0], conn[:, 1]
    a, E = aed[:, 0], aed[:, 1]
    d = joints[j1] - joints[j0]
    L = np.sqrt((d * d).sum(axis=1))
    c = d / L[:, None]
    k = E * a / L
    gm = N_m / L
    dp = phi[:, j1] - phi[:, j0]                         # [k, M, d]
    t = (c[None] * dp).sum(axis=2)                       # [k, M]
    s = (dp * dp).sum(axis=2)
    g1 = (g * lam)[:, None]                              # cotangent x lambda
    g2 = (g * lam * lam)[:, None]                        # cotangent x lambda^2
    t2 = t * t
    g_aed = np.stack([(g1 * (E / L) * t2).sum(0), (g1 * (a / L) * t2).sum(0), np.zeros(len(L))], axis=1)
    g_axial = (g2 * (s - t2) / L).sum(0)
    a2 = 2.0 * t[..., None] * dp - 3.0 * t2[..., None] * c[None]
    v = ((g1 * k / L)[..., None] * a2).sum(0) - ((g2 * gm / L)[..., None] * (a2 + s[..., None] * c[None])).sum(0)
    g_xyz = np.zeros((nJ, dim))
    np.add.at(g_xyz, j1, v)
    np.add.at(g_xyz, j0, -v)
    return g_xyz, g_aed, g_axial
