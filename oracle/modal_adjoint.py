"""numpy restatement of the reverse mode of the modal analysis, ``tb_modes_adjoint`` (TEST INFRASTRUCTURE ONLY).

``eigval_grad`` gives the gradients of L = sum_k g_k lambda_k for given eigenpairs (the oracle's from ``modal.modes`` or the
device's): dlambda/dp = phi^T (dK/dp - lambda dM/dp) phi per member, with the member geometry and the mass models of
``oracle/modal.py``.  It is checked against finite differences of ``modal.modes`` and a closed form
(tests/test_modes_adjoint_cpu.py); the CUDA kernel k_modes_sens is checked against it (tests/test_gpu_modes_adjoint.py).
"""
from __future__ import annotations

import numpy as np

from oracle import truss_oracle as orc


def eigval_grad(dim, joints, support, conn, aed, eigval, modes, g_eigval, consistent=False):
    """Gradients of L = sum_k g_eigval[k] eigval[k] for M-normalised eigenpairs (``modes`` [k, N], dense; entries at
    supported DOFs are ignored).  Returns (g_xyz [nJ, d], g_aed [M, 3], g_joint_mass [nJ]).

    Member m from j0 to j1: d = x_j1 - x_j0, L = |d|, c = d / L, k_m = E a / L, dphi = phi_j1 - phi_j0, t = c.dphi and w
    the mass quadratic form per unit member mass (lumped (|phi_j0|^2 + |phi_j1|^2) / 2, consistent
    (|phi_j0|^2 + |phi_j1|^2 + phi_j0.phi_j1) / 3):
      dlambda/da = (E/L) t^2 - lambda L rho w,  dlambda/dE = (a/L) t^2,  dlambda/drho = -lambda a L w,
      dlambda/dx_j1 = -dlambda/dx_j0 = (k_m/L) (2 t dphi - 3 t^2 c) - lambda rho a w c,
      dlambda/dmu_J = -lambda |phi_J|^2.
    Exact for simple eigenvalues; for a cluster only with a cotangent equal across it."""
    joints = np.asarray(joints, dtype=np.float64).reshape(-1, dim)
    conn = np.asarray(conn).astype(np.int64).reshape(-1, 2)
    aed = np.asarray(aed, dtype=np.float64).reshape(-1, 3)
    nJ = joints.shape[0]
    mask = orc.free_mask(dim, np.asarray(support))
    lam = np.asarray(eigval, dtype=np.float64).reshape(-1)
    g = np.asarray(g_eigval, dtype=np.float64).reshape(-1)
    phi = np.where(mask, np.asarray(modes, dtype=np.float64).reshape(len(lam), -1), 0.0).reshape(len(lam), nJ, dim)
    j0, j1 = conn[:, 0], conn[:, 1]
    a, E, rho = aed[:, 0], aed[:, 1], aed[:, 2]
    d = joints[j1] - joints[j0]
    L = np.sqrt((d * d).sum(axis=1))
    c = d / L[:, None]
    k = E * a / L
    p0, p1 = phi[:, j0], phi[:, j1]                      # [k, M, d]
    dp = p1 - p0
    t = (c[None] * dp).sum(axis=2)                       # [k, M]
    s = (p0 * p0).sum(axis=2) + (p1 * p1).sum(axis=2)
    w = (s + (p0 * p1).sum(axis=2)) / 3.0 if consistent else 0.5 * s
    gl = (g * lam)[:, None]
    g_aed = np.stack([(g[:, None] * (E / L) * t * t).sum(0) - (gl * L * rho * w).sum(0),
                      (g[:, None] * (a / L) * t * t).sum(0),
                      -(gl * a * L * w).sum(0)], axis=1)
    v = (g[:, None, None] * ((k / L)[None, :, None] * (2.0 * t[..., None] * dp - 3.0 * (t * t)[..., None] * c[None]))).sum(0) \
        - ((gl * rho * a * w)[..., None] * c[None]).sum(0)
    g_xyz = np.zeros((nJ, dim))
    np.add.at(g_xyz, j1, v)
    np.add.at(g_xyz, j0, -v)
    g_jm = -(gl[:, :, None] * phi * phi).sum(axis=(0, 2))
    return g_xyz, g_aed, g_jm
