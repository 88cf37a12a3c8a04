"""numpy restatement of the linear buckling analysis of ``tb_buckling`` (TEST INFRASTRUCTURE ONLY).

For a member-force state N (tension positive), the load factors lambda at which K_ff + lambda K_G,ff is singular:

  K_ff phi = lambda (-K_G,ff) phi,   K_ff from ``truss_oracle.assemble_K``

K_G is the transverse ("I - c c^T") form of the truss geometric stiffness: member m from j0 to j1 with direction cosines
c and length L (the static solve's ``member_length`` / ``member_cosines``) adds, with g = N_m / L,

  +g (delta_ij - c_i c_j) to the blocks (j0, j0) and (j1, j1),  -g (delta_ij - c_i c_j) to (j0, j1) and (j1, j0),

c_i c_j rounded as K's product, summed in ascending member order.  (The simpler (N/L) I differs from it by a term of
relative size N/(EA).)  nu = eig(K_G,ff, K_ff) by ``scipy.linalg.eigh(K_G_ff, K_ff)``, ascending; mode q is critical when
nu_q < -TAU max|nu| and then lambda_q = -1 / nu_q, else +inf with a zero mode row.  Modes are dense over the N DOFs
(0 at supports), K-normalised, with the component of largest magnitude positive.  The CUDA entry point ``tb_buckling``
is checked against this; this is checked against closed forms (tests/test_buckling_cpu.py).
"""
from __future__ import annotations

import numpy as np
import scipy.linalg as sl

from oracle import modal
from oracle import truss_oracle as orc

TAU = 1e-12   # relative threshold of a critical eigenvalue (BUCKLING_TAU in csrc/tb_modes.cu)


def geometric_stiffness(dim, joints, conn, axial) -> np.ndarray:
    """Dense N x N geometric stiffness over all DOFs (before the supports are removed)."""
    joints = np.asarray(joints, dtype=np.float64).reshape(-1, dim)
    conn = np.asarray(conn).astype(np.int64).reshape(-1, 2)
    axial = np.asarray(axial, dtype=np.float64).reshape(-1)
    N = joints.shape[0] * dim
    KG = np.zeros((N, N))
    for m, (j0, j1) in enumerate(conn):
        length = orc.member_length(joints[j0], joints[j1])
        c = orc.member_cosines(joints[j0], joints[j1], length)
        g = float(axial[m]) / length
        t = np.empty((dim, dim))
        for i in range(dim):
            for j in range(dim):
                t[i, j] = 1.0 - c[i] ** 2. if i == j else -(c[i] * c[j])
        blk = np.empty((2 * dim, 2 * dim))
        blk[:dim, :dim] = t
        blk[:dim, dim:] = -t
        blk[dim:, :dim] = -t
        blk[dim:, dim:] = t
        ke = g * blk
        for a, x in ((0, j0 * dim), (dim, j1 * dim)):
            for b, y in ((0, j0 * dim), (dim, j1 * dim)):
                KG[x:x + dim, y:y + dim] += ke[a:a + dim, b:b + dim]
    return KG


def buckling(dim, joints, support, conn, aed, axial, n_modes=None):
    """dict(nu [n] (ascending), factor [k], modes [k, N] (dense, K-normalised, zero rows for inf factors), K_ff, K_G_ff,
    mask)."""
    mask = orc.free_mask(dim, np.asarray(support))
    K = orc.assemble_K(dim, np.asarray(joints, dtype=np.float64).reshape(-1, dim), np.asarray(conn).reshape(-1, 2),
                       np.asarray(aed, dtype=np.float64).reshape(-1, 3))
    KG = geometric_stiffness(dim, joints, conn, axial)
    Kff, KGff = K[np.ix_(mask, mask)], KG[np.ix_(mask, mask)]
    nu, vec = sl.eigh(KGff, Kff)
    vec = vec / np.sqrt(np.einsum("ik,ij,jk->k", vec, Kff, vec))   # (eigh already K-normalises; made explicit)
    vec = modal.sign_normalise(vec)
    crit = nu < -TAU * (np.abs(nu).max() if nu.size else 0.0)
    with np.errstate(divide="ignore"):
        factor = np.where(crit, -1.0 / np.where(crit, nu, -1.0), np.inf)
    k = len(nu) if n_modes is None else int(n_modes)
    dense = np.zeros((k, mask.shape[0]))
    dense[:, mask] = (vec[:, :k] * crit[:k]).T
    return {"nu": nu, "factor": factor[:k], "factor_all": factor, "modes": dense, "critical": crit, "K_ff": Kff,
            "K_G_ff": KGff, "mask": mask}
