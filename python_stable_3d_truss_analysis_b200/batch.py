"""Batched entry points next to the reference's one-truss-at-a-time API.

The reference solves exactly one truss per ``Truss.Solve()`` call and its callers loop in Python
(``ga.py:155-160`` over genes, ``generate.py:342-357`` over generated trusses).  These functions
hand the whole batch to the CUDA library in one call:

  ``SolveBatch(trusses)``                    any list of Truss objects (shared or ragged topology)
  ``SolveLoadCases(truss, forces)``          one truss, many dense load vectors (same K, many f)
  ``SolveMemberTypes(truss, genes, types)``  one truss, many member-type assignments (GA population)
  ``FitnessBatch(...)``                      GA.GetFitness for a population (ga.py:139-149)
  ``SolveWithFixedMemberType(trusses, t)``   the graph-data converter's double solve (data.py:17-44, 108-114)
  ``ModesBatch(truss, ...)``                 natural frequencies and mode shapes of many sizings of one truss
  ``SolveModesBatch(trusses, ...)``          natural frequencies and mode shapes of trusses of any topologies
  ``BucklingBatch(truss, ...)``              critical load factors and buckling modes of many sizings of one truss

All of them return dense numpy arrays (``u [B,N]``, ``ext [B,N]``, ``axial [B,M]``, ``weight [B]``,
``info [B]``); ``SolveBatch`` also stores the results back into the Truss objects.
"""
from __future__ import annotations

import numpy as np

from . import _lib
from .truss import ZERO_EPS, Truss, make_plan, raise_for_info, raise_for_modes_info
from .type import MemberType


def type_table(memberTypeList):
    """[T,3] float64 (a, e, density) table from MemberType objects or triples."""
    return np.array([t.Serialize() if isinstance(t, MemberType) else list(t) for t in memberTypeList],
                    dtype=np.float64).reshape(-1, 3)


def _check_infos(info, raise_on_error):
    if raise_on_error:
        bad = np.nonzero(info)[0]
        if bad.size:
            raise_for_info(int(info[bad[0]]))


def SolveLoadCases(truss: Truss, forces, raise_on_error=True, independent=False):
    """One truss under B load cases.  ``forces`` is [B, N] dense (index jointID*dim + axis).

    Equivalent to ``for f in forces: truss.SetForces(f); truss.Solve()`` (truss.py:329-364).  The stiffness matrix is the
    same for every load case, so on the band path it is assembled and factorised once (tb_solve_loadcases_host) when
    the member products fit shared memory (else every load case is factorised on its own);
    ``independent=True`` factorises every system on its own, as a batch of unrelated trusses would (tb_solve_host)."""
    xyz, support, conn, aed, _ = truss._pack()
    forces = np.ascontiguousarray(forces, dtype=np.float64).reshape(-1, truss.nJoint * truss.dim)
    plan = truss._get_plan(support, conn)
    out = plan.solve_host(forces.shape[0], xyz, forces, aed=aed, shared_factor=not independent)
    _check_infos(out["info"], raise_on_error)
    return out


def SolveMemberTypes(truss: Truss, genes, memberTypeList, raise_on_error=True):
    """One truss under B member-type assignments; ``genes`` is int [B, M] of indices into the list."""
    xyz, support, conn, _, force = truss._pack()
    genes = np.ascontiguousarray(genes, dtype=np.int32).reshape(-1, truss.nMember)
    plan = truss._get_plan(support, conn)
    out = plan.solve_host(genes.shape[0], xyz, force, gene=genes, type_table=type_table(memberTypeList))
    _check_infos(out["info"], raise_on_error)
    return out


def FitnessBatch(truss: Truss, genes, memberTypeList, allowStress, allowDisplace, full=False):
    """GA.GetFitness (ga.py:139-149) for a whole population in one call.

    Returns dict(fitness [B], flags [B,2] (stress ok, displacement ok), info [B]) (+ full results)."""
    xyz, support, conn, _, force = truss._pack()
    genes = np.ascontiguousarray(genes, dtype=np.int32).reshape(-1, truss.nMember)
    plan = truss._get_plan(support, conn)
    return plan.fitness_host(genes.shape[0], xyz, force, genes, type_table(memberTypeList), allowStress,
                             allowDisplace, full=full)


def ModesBatch(truss: Truss, aed=None, genes=None, memberTypeList=None, nMode=None, isConsistentMass=False,
               jointMasses=None, raise_on_error=True, want_modes=True):
    """Modal analysis of B sizings of one truss in one call (tb_modes_host): ``Truss.SolveModes`` per design, e.g. the
    frequency constraints of a GA population.  Member properties are either explicit, ``aed`` [B, M, 3] (a, e, density),
    or ``genes`` int [B, M] of indices into ``memberTypeList``.  ``jointMasses``: {jointID: mass} shared by the batch, or
    an array [nJ] / [B, nJ].  Returns dict(eigval [B, k] (lambda = omega^2, ascending), modes [B, k, N] (M-normalised, 0
    at supported DOFs), info [B]); ``nMode=None`` = all modes."""
    xyz, support, conn, _, _ = truss._pack()
    plan = truss._get_plan(support, conn)
    jm = jointMasses
    if isinstance(jointMasses, dict):
        jm = np.zeros(truss.nJoint)
        for j, mass in jointMasses.items():
            jm[j] = float(mass)
    if (aed is None) == (genes is None):
        raise ValueError("give either aed or genes (with memberTypeList)")
    if aed is not None:
        aed = np.ascontiguousarray(aed, dtype=np.float64).reshape(-1, truss.nMember * 3)
        out = plan.modes_host(aed.shape[0], xyz, aed=aed, n_modes=nMode, consistent=isConsistentMass, joint_mass=jm,
                              want_modes=want_modes)
    else:
        genes = np.ascontiguousarray(genes, dtype=np.int32).reshape(-1, truss.nMember)
        out = plan.modes_host(genes.shape[0], xyz, gene=genes, type_table=type_table(memberTypeList), n_modes=nMode,
                              consistent=isConsistentMass, joint_mass=jm, want_modes=want_modes)
    if raise_on_error:
        bad = np.nonzero(out["info"])[0]
        if bad.size:
            raise_for_modes_info(int(out["info"][bad[0]]))
    return out


def BucklingBatch(truss: Truss, aed=None, genes=None, memberTypeList=None, nMode=None, raise_on_error=True,
                  want_modes=True):
    """Linear buckling of B sizings of one truss under its loads (``Truss.SolveBuckling`` per design, e.g. a stability
    constraint on a GA population): one static call (tb_solve_host) for the member forces, then one buckling call
    (tb_buckling_host) with them.  Member properties are either explicit, ``aed`` [B, M, 3] (a, e, density), or
    ``genes`` int [B, M] of indices into ``memberTypeList``.  Returns dict(factor [B, k] (load factors ascending, inf for
    modes no positive multiple of the loads reaches), modes [B, k, N] (K-normalised, 0 at supported DOFs and for inf
    factors; with ``want_modes``), axial [B, M] (the member forces of the static solve), info [B] (the buckling call's:
    it fails where the static solve does)); ``nMode=None`` = one per free DOF."""
    xyz, support, conn, _, force = truss._pack()
    plan = truss._get_plan(support, conn)
    if (aed is None) == (genes is None):
        raise ValueError("give either aed or genes (with memberTypeList)")
    if aed is not None:
        aed = np.ascontiguousarray(aed, dtype=np.float64).reshape(-1, truss.nMember * 3)
        props = dict(aed=aed)
        B = aed.shape[0]
    else:
        genes = np.ascontiguousarray(genes, dtype=np.int32).reshape(-1, truss.nMember)
        props = dict(gene=genes, type_table=type_table(memberTypeList))
        B = genes.shape[0]
    st = plan.solve_host(B, xyz, force, want=("axial",), **props)
    out = plan.buckling_host(B, xyz, st["axial"], n_modes=nMode, want_modes=want_modes, **props)
    out["axial"] = st["axial"]
    if raise_on_error:
        bad = np.nonzero(out["info"])[0]
        if bad.size:
            raise_for_modes_info(int(out["info"][bad[0]]))
    return out


def SolveModesBatch(trusses, nMode=None, isConsistentMass=False, jointMasses=None, raise_on_error=True):
    """``Truss.SolveModes`` for a list of Truss objects of any topologies in one ragged call (tb_modes_ragged_host); the
    results are stored into each truss (``GetEigenvalues`` / ``GetNaturalFrequencies`` / ``GetModeShapes``).
    ``nMode``: modes per truss, None = all modes of each truss (an ``nMode`` above a truss's free-DOF count raises, as
    ``Truss.SolveModes`` does).  ``jointMasses``: None or one {jointID: mass} dict (or None) per truss.  Returns the
    per-truss info codes; a failed truss keeps no modes (``raise_on_error`` raises for the first one)."""
    trusses = list(trusses)
    if not trusses:
        return np.zeros(0, np.int32)
    dim = trusses[0].dim
    if any(t.dim != dim for t in trusses):
        raise ValueError("all trusses of a batch must have the same dimension")
    if jointMasses is not None and len(jointMasses) != len(trusses):
        raise ValueError(f"jointMasses must hold one entry per truss ({len(trusses)}), not {len(jointMasses)}")
    dim, jo, mo, xyz, sup, conn, aed, _ = pack_ragged(trusses)
    cs = np.concatenate([[0], np.cumsum(_lib.free_dofs_per_joint(dim, sup))])
    n_free = cs[jo[1:]] - cs[jo[:-1]]
    if nMode is not None:
        nMode = int(nMode)
        short = np.nonzero(n_free < nMode)[0]
        if nMode < 1 or short.size:
            i = int(short[0]) if short.size else 0
            raise ValueError(f"nMode = {nMode} is not in [1, {int(n_free[i])}], the free DOFs of truss {i}")
    jm = None
    if jointMasses is not None and any(jointMasses):
        jm = np.zeros(int(jo[-1]))
        for i, (t, masses) in enumerate(zip(trusses, jointMasses)):
            for j, mass in (masses or {}).items():
                if not 0 <= int(j) < t.nJoint:
                    raise ValueError(f"truss {i}: no such joint [{j}], can't add a mass on it")
                jm[jo[i] + int(j)] = float(mass)
    k = int(n_free.max(initial=0)) if nMode is None else nMode
    k = min(max(k, 1), 160)
    out = _lib.modes_ragged_host(dim, jo, mo, xyz, sup, conn, aed, k, consistent=isConsistentMass, joint_mass=jm)
    for i, t in enumerate(trusses):
        if out["info"][i] != 0:
            continue
        q = int(out["n_free"][i]) if nMode is None else nMode
        N = dim * int(jo[i + 1] - jo[i])
        block = out["modes"][k * dim * jo[i]:k * dim * jo[i + 1]].reshape(k, N)
        t._modes = {"eigval": out["eigval"][i, :q].copy(), "modes": block[:q].copy()}
    if raise_on_error:
        bad = np.nonzero(out["info"])[0]
        if bad.size:
            raise_for_modes_info(int(out["info"][bad[0]]))
    return out["info"]


def pack_ragged(trusses):
    """Pack Truss objects back to back in the tb_ragged_in layout."""
    dim = trusses[0].dim
    packs = [t._pack() for t in trusses]
    joint_off = np.zeros(len(trusses) + 1, np.int64)
    member_off = np.zeros(len(trusses) + 1, np.int64)
    joint_off[1:] = np.cumsum([p[0].shape[0] for p in packs])
    member_off[1:] = np.cumsum([p[2].shape[0] for p in packs])
    cat = lambda i, dt: np.concatenate([np.asarray(p[i]).reshape(-1) for p in packs]).astype(dt)  # noqa: E731
    return dim, joint_off, member_off, cat(0, np.float64), cat(1, np.uint8), cat(2, np.int32), cat(3, np.float64), \
        cat(4, np.float64)


_PLAN_CACHE = {}


def _cached_plan(dim, conn, support):
    """Plans of the last few topologies seen by the batched calls (a plan costs a host pass over the scatter map and a
    few uploads; repeated batches of one topology should not pay it again)."""
    key = (dim, conn.shape[0], support.tobytes(), conn.tobytes())
    plan = _PLAN_CACHE.pop(key, None)
    if plan is None:
        plan = make_plan(dim, conn, support)
    _PLAN_CACHE[key] = plan                     # (re-inserted: most recently used last)
    while len(_PLAN_CACHE) > 8:
        _PLAN_CACHE.pop(next(iter(_PLAN_CACHE)))
    return plan


def _solve_packs(dim, packs):
    """Dense results of a list of packed trusses ((xyz, support, conn, aed, force) each): same topology everywhere -> one
    plan and a uniform batch per topology group; otherwise, if every truss fits the fused shared-memory kernel, one ragged
    batch (the generator's case).  Returns (u, ext, axial) as lists of per-truss arrays and the info codes."""
    n = len(packs)
    info = np.zeros(n, np.int32)
    u, ext, axial = [None] * n, [None] * n, [None] * n

    def signature(p):
        return (p[0].shape[0], p[2].shape[0], p[1].tobytes(), p[2].tobytes())

    groups = {}
    for i, p in enumerate(packs):
        groups.setdefault(signature(p), []).append(i)

    # one ragged batch needs the LARGEST truss of the batch to fit the fused kernels' shared memory
    fits_small = _lib.small_path_fits(dim, max(p[0].shape[0] for p in packs), max(p[2].shape[0] for p in packs))
    if len(groups) > 1 and fits_small:
        joint_off = np.zeros(n + 1, np.int64)
        member_off = np.zeros(n + 1, np.int64)
        joint_off[1:] = np.cumsum([p[0].shape[0] for p in packs])
        member_off[1:] = np.cumsum([p[2].shape[0] for p in packs])
        cat = lambda i, dt: np.concatenate([np.asarray(p[i]).reshape(-1) for p in packs]).astype(dt)  # noqa: E731
        out = _lib.solve_ragged_host(dim, joint_off, member_off, cat(0, np.float64), cat(1, np.uint8), cat(2, np.int32),
                                     cat(3, np.float64), cat(4, np.float64), want=("u", "ext", "axial"))
        for i in range(n):
            info[i] = out["info"][i]
            u[i] = out["u"][joint_off[i] * dim:joint_off[i + 1] * dim]
            ext[i] = out["ext"][joint_off[i] * dim:joint_off[i + 1] * dim]
            axial[i] = out["axial"][member_off[i]:member_off[i + 1]]
    else:
        for idx in groups.values():
            p0 = packs[idx[0]]
            plan = _cached_plan(dim, p0[2], p0[1])
            out = plan.solve_host(len(idx), np.stack([packs[i][0] for i in idx]), np.stack([packs[i][4] for i in idx]),
                                  aed=np.stack([packs[i][3] for i in idx]), want=("u", "ext", "axial"))
            for k, i in enumerate(idx):
                info[i] = out["info"][k]
                u[i], ext[i], axial[i] = out["u"][k], out["ext"][k], out["axial"][k]
    return u, ext, axial, info


def SolveBatch(trusses, raise_on_error=True):
    """Solve a list of Truss objects in one call and store the results into them.

    Same topology everywhere -> one plan, uniform batch.  Otherwise, if every truss fits the fused
    shared-memory kernel, one ragged batch (the generator's case); else grouped by topology.
    Returns the per-truss info codes."""
    trusses = list(trusses)
    if not trusses:
        return np.zeros(0, np.int32)
    dim = trusses[0].dim
    if any(t.dim != dim for t in trusses):
        raise ValueError("all trusses of a batch must have the same dimension")
    u, ext, axial, info = _solve_packs(dim, [t._pack() for t in trusses])
    for i, t in enumerate(trusses):
        if info[i] == 0:
            t._set_dense_results(u[i], ext[i], axial[i])
    _check_infos(info, raise_on_error)
    return info


def SolveWithFixedMemberType(trusses, fixedMemberType=MemberType(1., 1e7, 0.1), raise_on_error=True, dense=False):
    """The double solve of the reference's graph-data converter for a whole list of trusses in two batched calls.

    ``TrussHeteroDataCreator.FromTruss`` / ``FromJSON`` (data.py:17-44) solve the truss as it is and then, in
    ``__GetFixedInternalAndDisplace`` (data.py:108-114), copy it, set EVERY member to ``fixedMemberType`` and solve again
    to get reference stresses and displacements that do not depend on the member sizing.  Here the trusses that are not
    solved yet go through ``SolveBatch`` and the fixed-type variants through a second batch that reuses the same packed
    arrays with the member properties replaced -- no Truss copies.

    Returns a list of ``(fixedInternals, fixedDisplaces)`` per truss, the reference's dicts
    (``GetInternalStresses()`` = force / area over the members with |force| >= 1e-10, ``GetDisplacements()`` over the
    joints with a non-zero displacement); with ``dense=True`` a dict of arrays instead:
    ``stress`` list of [M], ``u`` list of [N], ``info`` [B]."""
    trusses = list(trusses)
    if not trusses:
        return {"stress": [], "u": [], "info": np.zeros(0, np.int32)} if dense else []
    dim = trusses[0].dim
    todo = [t for t in trusses if not t.isSolved]
    if todo:
        SolveBatch(todo, raise_on_error=raise_on_error)
    fixed = np.asarray(fixedMemberType.Serialize() if isinstance(fixedMemberType, MemberType) else fixedMemberType,
                       dtype=np.float64).reshape(3)
    packs = []
    for t in trusses:
        xyz, support, conn, aed, force = t._pack()
        packs.append((xyz, support, conn, np.broadcast_to(fixed, aed.shape).copy(), force))
    u, _, axial, info = _solve_packs(dim, packs)
    _check_infos(info, raise_on_error)
    stress = [a / fixed[0] for a in axial]
    if dense:
        return {"stress": stress, "u": u, "info": info}
    out = []
    for i in range(len(trusses)):
        if info[i] != 0:
            out.append((None, None))
            continue
        ax, rows = axial[i], np.asarray(u[i]).reshape(-1, dim)
        internals = {int(m): float(ax[m]) / float(fixed[0]) for m in np.nonzero(~(np.abs(ax) < ZERO_EPS))[0]}
        displaces = {int(j): rows[j].copy() for j in np.nonzero(~(np.abs(rows) < ZERO_EPS).all(axis=1))[0]}
        out.append((internals, displaces))
    return out
