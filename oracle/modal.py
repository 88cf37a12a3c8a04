"""numpy restatement of the modal analysis of ``tb_modes`` (TEST INFRASTRUCTURE ONLY).

Free vibration K_ff phi = lambda M_ff phi over the free DOFs (supported DOFs dropped in the reference's mask order),
with K_ff from ``truss_oracle.assemble_K`` and the mass from the same member geometry:

  member mass   m_e = (a L) density, the weight term's product and rounding (truss.py:52-54, 166-168)
  lumped        m_e / 2 on every axis of both end joints
  consistent    (m_e / 6) [[2, 1], [1, 2]] per member and axis over its two end joints
  joint_mass    a non-structural mass on every axis of its joint (both models)

Eigenpairs by ``scipy.linalg.eigh(K_ff, M_ff)``; mode shapes are dense over the N DOFs (0 at supports), M-normalised,
with the component of largest magnitude positive (on a tie the lowest index).  The CUDA entry point ``tb_modes`` is
checked against this; this is checked against closed forms (tests/test_modes_cpu.py).
"""
from __future__ import annotations

import numpy as np
import scipy.linalg as sl

from oracle import truss_oracle as orc


def member_masses(dim, joints, conn, aed) -> np.ndarray:
    """m_e = (a * L) * density per member."""
    joints = np.asarray(joints, dtype=np.float64).reshape(-1, dim)
    out = np.zeros(len(conn))
    for m, ((j0, j1), (a, _e, rho)) in enumerate(zip(np.asarray(conn).reshape(-1, 2), np.asarray(aed).reshape(-1, 3))):
        out[m] = (a * orc.member_length(joints[j0], joints[j1])) * rho
    return out


def mass_matrix(dim, joints, conn, aed, consistent=False, joint_mass=None) -> np.ndarray:
    """Dense N x N mass matrix over all DOFs (before the supports are removed)."""
    joints = np.asarray(joints, dtype=np.float64).reshape(-1, dim)
    conn = np.asarray(conn).astype(np.int64).reshape(-1, 2)
    nJ = joints.shape[0]
    N = nJ * dim
    Mm = np.zeros((N, N))
    me = member_masses(dim, joints, conn, aed)
    for m, (j0, j1) in enumerate(conn):
        for ax in range(dim):
            a, b = j0 * dim + ax, j1 * dim + ax
            if consistent:
                m6 = me[m] / 6.0
                Mm[a, a] += 2.0 * m6
                Mm[b, b] += 2.0 * m6
                Mm[a, b] += m6
                Mm[b, a] += m6
            else:
                Mm[a, a] += me[m] * 0.5
                Mm[b, b] += me[m] * 0.5
    if joint_mass is not None:
        Mm[np.diag_indices(N)] += np.repeat(np.asarray(joint_mass, dtype=np.float64).reshape(nJ), dim)
    return Mm


def reduced(dim, joints, support, conn, aed, consistent=False, joint_mass=None):
    """(K_ff, M_ff, free mask)."""
    mask = orc.free_mask(dim, np.asarray(support))
    K = orc.assemble_K(dim, joints, conn, aed)
    Mm = mass_matrix(dim, joints, conn, aed, consistent, joint_mass)
    return K[np.ix_(mask, mask)], Mm[np.ix_(mask, mask)], mask


def sign_normalise(phi: np.ndarray) -> np.ndarray:
    """Columns of phi (any leading shape [n, k]) flipped so that the component of largest magnitude is positive; np.argmax
    returns the lowest index on a tie."""
    phi = np.array(phi, dtype=np.float64, copy=True)
    idx = np.argmax(np.abs(phi), axis=0)
    s = np.where(phi[idx, np.arange(phi.shape[1])] < 0.0, -1.0, 1.0)
    return phi * s


def modes(dim, joints, support, conn, aed, consistent=False, joint_mass=None, n_modes=None):
    """dict(eigval [k], modes [k, N] (dense, M-normalised, sign convention), eigval_all [n], K_ff, M_ff, mask)."""
    Kff, Mff, mask = reduced(dim, joints, support, conn, aed, consistent, joint_mass)
    lam, vec = sl.eigh(Kff, Mff)
    vec = vec / np.sqrt(np.einsum("ik,ij,jk->k", vec, Mff, vec))   # (eigh already M-normalises; made explicit)
    vec = sign_normalise(vec)
    k = len(lam) if n_modes is None else int(n_modes)
    N = mask.shape[0]
    dense = np.zeros((k, N))
    dense[:, mask] = vec[:, :k].T
    return {"eigval": lam[:k], "modes": dense, "eigval_all": lam, "K_ff": Kff, "M_ff": Mff, "mask": mask}


def clusters(lam, rel=1e-6):
    """Index groups of eigenvalues whose neighbours are closer than rel * max|lambda| (ascending lam)."""
    lam = np.asarray(lam)
    scale = np.max(np.abs(lam)) if lam.size else 1.0
    groups, cur = [], [0]
    for i in range(1, len(lam)):
        if lam[i] - lam[i - 1] <= rel * scale:
            cur.append(i)
        else:
            groups.append(cur)
            cur = [i]
    if lam.size:
        groups.append(cur)
    return groups
