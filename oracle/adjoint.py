"""numpy restatement of the reverse mode of ``Truss.Solve()`` (TEST INFRASTRUCTURE ONLY).

Given the cotangents of the solve's outputs (``u`` [N], ``ext`` [N], ``axial`` [M], ``weight``), returns the gradients
of the scalar they define with respect to the joint coordinates, the member properties (a, e, density) and the load
vector, by one adjoint solve with the same reduced stiffness matrix (DESIGN.md section 9).  The CUDA entry point
``tb_adjoint`` is checked against this; this is checked against central differences of ``truss_oracle.solve``.
"""
from __future__ import annotations

import numpy as np

from oracle import truss_oracle as orc


def adjoint(dim, joints, support, conn, aed, force, g_u=None, g_ext=None, g_axial=None, g_w=0.0):
    """Returns dict(joint_xyz [nJ, dim], member_aed [M, 3], force [N], lam [N], u [N])."""
    joints = np.asarray(joints, dtype=np.float64).reshape(-1, dim)
    conn = np.asarray(conn).astype(np.int64).reshape(-1, 2)
    aed = np.asarray(aed, dtype=np.float64).reshape(-1, 3)
    nJ, M = joints.shape[0], conn.shape[0]
    N = nJ * dim
    g_u = np.zeros(N) if g_u is None else np.asarray(g_u, dtype=np.float64).reshape(N)
    g_ext = np.zeros(N) if g_ext is None else np.asarray(g_ext, dtype=np.float64).reshape(N)
    g_axial = np.zeros(M) if g_axial is None else np.asarray(g_axial, dtype=np.float64).reshape(M)
    mask = orc.free_mask(dim, support)
    K = orc.assemble_K(dim, joints, conn, aed)
    Kff = K[np.ix_(mask, mask)]
    f = np.asarray(force, dtype=np.float64).reshape(N)
    u = np.zeros(N)
    u[mask] = np.linalg.solve(Kff, f[mask])

    j0, j1 = conn[:, 0], conn[:, 1]
    d = joints[j1] - joints[j0]                                       # [M, dim]
    L = np.sqrt((d ** 2).sum(axis=1))
    c = d / L[:, None]
    A, E, rho = aed[:, 0], aed[:, 1], aed[:, 2]
    k = E * A / L
    J = lambda v: v.reshape(nJ, dim)                                  # noqa: E731
    delta = lambda v: J(v)[j1] - J(v)[j0]                             # noqa: E731

    # 1. total cotangent of the member forces: the axial one plus the reactions' (linear in N)
    z = np.where(mask, 0.0, g_ext)
    n_hat = g_axial + (c * delta(z)).sum(axis=1)
    # 2. adjoint load, 3. adjoint solve with the forward's K_ff
    r = J(g_u.copy())
    P = (n_hat * k)[:, None] * c
    np.add.at(r, j1, P)
    np.add.at(r, j0, -P)
    r = r.reshape(N)
    lam = np.zeros(N)
    lam[mask] = np.linalg.solve(Kff, r[mask])
    # 4. member properties
    du, dlam, dz = delta(u), delta(lam), delta(z)
    tu = (c * du).sum(axis=1)
    q = n_hat - (c * dlam).sum(axis=1)
    g_aed = np.stack([E / L * tu * q + g_w * L * rho, A / L * tu * q, g_w * A * L], axis=1)
    # 5. loads: the free ones, through lambda and through ext = f there
    g_f = np.where(mask, lam + g_ext, 0.0)
    # 6. geometry: gradient with respect to d = x_j1 - x_j0 of s [g_axial (d.du)/L^2 + (d.dw)(d.du)/L^3] + g_w A rho L
    dw = dz - dlam
    tw = (c * dw).sum(axis=1)
    G = (k / L)[:, None] * (g_axial[:, None] * (du - 2.0 * tu[:, None] * c) + dw * tu[:, None] + du * tw[:, None]
                            - 3.0 * (tu * tw)[:, None] * c) + (g_w * A * rho)[:, None] * c
    g_x = np.zeros((nJ, dim))
    np.add.at(g_x, j1, G)
    np.add.at(g_x, j0, -G)
    return {"joint_xyz": g_x, "member_aed": g_aed, "force": g_f, "lam": lam, "u": u}


def loss(out, g_u=None, g_ext=None, g_axial=None, g_w=0.0):
    """The scalar the cotangents define: <g_u, u> + <g_ext, ext> + <g_axial, axial> + g_w * weight."""
    s = g_w * out["weight"]
    for g, k in ((g_u, "u"), (g_ext, "ext"), (g_axial, "axial")):
        if g is not None:
            s += float(np.dot(np.ravel(g), np.ravel(out[k])))
    return s
