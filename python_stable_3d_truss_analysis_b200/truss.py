"""``Truss`` / ``Member`` -- the reference's solver-facing API on top of the CUDA library.

Drop-in for ``slientruss3d/truss.py`` (``Member :10-106``, ``Truss :109-466``; documented in
``detail/how_to_use.md:56-459`` and ``detail/combine_with_JSON.md:71-163``): same constructors,
builders, setters, getters, JSON layout and exceptions.  ``Truss.Solve()`` (``truss.py:329-364``)
packs the truss into flat arrays and runs it as a batch of one through ``libtruss_b200.so``;
there is no numpy/LAPACK solve here and no CPU fallback.  Results are kept dense; the sparse
dicts the reference exposes (entries with ``|x| >= 1e-10``, ``truss.py:344-361``) are built on
first access.

Deliberate differences from the reference (DESIGN.md "Reference quirks"):
  * ``AddNewMember`` stores its own copy of the ``MemberType`` -- the reference aliases the
    caller's instance, so ``SetMemberType`` on one member silently rewrites every member built
    from it (``truss.py:18,44-46``);
  * ``SetSupportType(s)`` work (the reference assigns into a tuple and always raises, ``:198-203``);
  * a stiffness matrix that is not positive definite raises ``numpy.linalg.LinAlgError`` with the
    failing leading minor instead of returning unchecked LU output.
"""
from __future__ import annotations

import copy
import json
from pprint import pformat

import numpy as np

from . import _lib
from .type import MemberType, SupportType
from .utils import (CheckDim, DimensionError, InvaildJointError, IsZero, IsZeroVector, GetLength, NotAllBeSetError,
                    TrussNotSolvedError, TrussNotStableError, ZERO_EPS)

INFO_NOT_STABLE, INFO_ZERO_LENGTH, INFO_BAD_SUPPORT, INFO_BAD_INDEX = -1, -2, -3, -4
INFO_MASS, INFO_NO_CONVERGENCE = _lib.TB_INFO_MASS, _lib.TB_INFO_NO_CONVERGENCE   # tb_modes only


class MassNotPositiveDefiniteError(ValueError):
    """Modal analysis: the reduced mass matrix is not positive definite (a free DOF without mass)."""


class ModesNotConvergedError(RuntimeError):
    """Modal analysis: the tridiagonal QL iteration hit its cap."""


def raise_for_modes_info(info: int):
    """Map a per-system status code of tb_modes onto an exception (the static solve's codes as raise_for_info)."""
    if info == INFO_MASS:
        raise MassNotPositiveDefiniteError("Mass matrix is not positive definite: a free DOF has no positive mass "
                                           "(give its members a density or its joint a joint mass)")
    if info == INFO_NO_CONVERGENCE:
        raise ModesNotConvergedError("The eigenvalue iteration did not converge")
    raise_for_info(info)


def raise_for_info(info: int):
    """Map a per-system status code of the C ABI onto the exception the reference would raise."""
    if info == 0:
        return
    if info == INFO_NOT_STABLE:
        raise TrussNotStableError("The truss is not stable !")
    if info == INFO_ZERO_LENGTH:
        raise ZeroDivisionError("float division by zero (a member has zero length)")
    if info == INFO_BAD_SUPPORT:
        from .utils import InvalidSupportTypeError
        raise InvalidSupportTypeError("[GetResistanceMask] No such support type !")
    if info == INFO_BAD_INDEX:
        raise InvaildJointError("A member refers to a joint (or member type) that does not exist.")
    raise np.linalg.LinAlgError(f"Stiffness matrix is not positive definite (leading minor {info}): "
                                "the truss is a mechanism or K is singular")


class Member:
    def __init__(self, joint0, joint1, dim=3, memberType=None):
        self._dim = CheckDim(dim)
        if len(joint0) != dim or len(joint1) != dim:
            raise DimensionError(f"Dimension of each joint must be {dim}, but got dim(joint0) = {len(joint0)} "
                                 f"and dim(joint1) = {len(joint1)}.")
        self._ends = [joint0, joint1]
        self._type = MemberType() if memberType is None else memberType
        self._refresh_length()

    def _refresh_length(self):
        p, q = self._ends
        self._length = sum((q[i] - p[i]) ** 2. for i in range(self._dim)) ** 0.5

    def __repr__(self):
        return f"Member[{self._ends[0]}, {self._ends[1]}, k={self.e * self.a / self._length :.4f}]"

    dim = property(lambda self: self._dim)
    e = property(lambda self: self._type.e)
    a = property(lambda self: self._type.a)
    density = property(lambda self: self._type.density)
    length = property(lambda self: self._length)

    @property
    def memberType(self):
        return self._type.Copy()

    @memberType.setter
    def memberType(self, other):
        self._type.Set(other)

    @property
    def weight(self):
        return self.a * self._length * self.density

    @property
    def k(self):
        return self.e * self.a / self._length

    @property
    def cosines(self):
        p, q = self._ends
        return [(q[i] - p[i]) / self._length for i in range(self._dim)]

    @property
    def matK(self):
        """Element stiffness in global axes, 2d x 2d (inspection helper; Solve() does not use it)."""
        c = np.array(self.cosines)
        cc = np.outer(c, c)
        return self.k * np.block([[cc, -cc], [-cc, cc]])

    def IsTension(self, forceVec):
        axis = np.array(self._ends[1]) - np.array(self._ends[0])
        return np.dot(axis, forceVec) > 0

    def SetPosition(self, jointID_0or1, position):
        if jointID_0or1 not in (0, 1):
            raise KeyError("[jointID_0or1] must be 0 or 1.")
        self._ends[jointID_0or1] = position
        self._refresh_length()

    def Serialize(self):
        return {"joint0": list(self._ends[0]), "joint1": list(self._ends[1]), "memberType": self._type.Serialize()}

    def Copy(self):
        return Member(tuple(self._ends[0]), tuple(self._ends[1]), self._dim, self._type.Copy())


def make_plan(dim, conn, support):
    """C-ABI plan of a topology, with the reference's exceptions for what tb_plan_create refuses (type.py:37-74 support
    codes, truss.py:252-254 joints of a member)."""
    support = np.asarray(support)
    if support.size and (support.min() < 0 or support.max() > SupportType.ROLLER_Z):
        from .utils import InvalidSupportTypeError
        raise InvalidSupportTypeError(f"[GetResistanceMask] No such {dim}D-support type !")
    try:
        return _lib.Plan(dim, conn, support.astype(np.uint8))
    except _lib.TrussLibError as exc:
        if exc.code == -5:
            from .utils import InvalidSupportTypeError
            raise InvalidSupportTypeError(f"[GetResistanceMask] No such {dim}D-support type !") from None
        if exc.code == -4:
            raise InvaildJointError("A member refers to a joint that does not exist.") from None
        raise


class Truss:
    def __init__(self, dim):
        self._dim = CheckDim(dim)
        self._joints = {}     # jointID  -> (position tuple, supportType)
        self._forces = {}     # jointID  -> force tuple
        self._members = {}    # memberID -> (jointID0, jointID1, Member)
        self._plan = None     # cached C-ABI plan of the current topology
        self._clear_results()

    # ------------------------------------------------------------------ internal state
    def _clear_results(self):
        self._dense = None                      # dict(u, ext, axial) of dense float64 arrays
        self._displace = self._external = self._internal = None
        self._solved = False
        self._modes = None                      # dict(eigval [k], modes [k, N]) of SolveModes()
        self._buckling = None                   # dict(factor [k], modes [k, N]) of SolveBuckling()

    def _topology_changed(self):
        self._plan = None
        self._modes = None
        self._buckling = None

    def _pack(self):
        """Flat arrays in the layout of include/truss_b200.h."""
        d, nj, nm = self._dim, len(self._joints), len(self._members)
        xyz = np.array([self._joints[j][0] for j in range(nj)], dtype=np.float64).reshape(nj, d)
        support = np.array([self._joints[j][1] for j in range(nj)], dtype=np.int64)
        conn = np.array([self._members[m][:2] for m in range(nm)], dtype=np.int32).reshape(nm, 2)
        aed = np.array([self._members[m][2]._type.Serialize() for m in range(nm)], dtype=np.float64).reshape(nm, 3)
        force = np.zeros((nj, d))
        for j, vec in self._forces.items():
            force[j] = vec
        return xyz, support, conn, aed, force.reshape(-1)

    def _get_plan(self, support=None, conn=None):
        if self._plan is None:
            if support is None:
                _, support, conn, _, _ = self._pack()
            self._plan = make_plan(self._dim, conn, support)
        return self._plan

    def _set_dense_results(self, u, ext, axial):
        self._dense = {"u": np.asarray(u, dtype=np.float64), "ext": np.asarray(ext, dtype=np.float64),
                       "axial": np.asarray(axial, dtype=np.float64)}
        self._displace = self._external = self._internal = None
        self._solved = True

    def _dense_or_from_sparse(self, key):
        """Dense result array ``key`` (u | ext | axial), rebuilt from the sparse dicts when the truss was loaded from an
        output JSON (the entries the reference dropped under its 1e-10 filter come back as zeros)."""
        if self._dense is not None:
            return np.asarray(self._dense[key], dtype=np.float64).reshape(-1)
        d = self._dim
        if key == "axial":
            v = np.zeros(self.nMember)
            for m, f in (self._internal or {}).items():
                v[m] = f
            return v
        v = np.zeros(self.nJoint * d)
        for j, vec in ((self._displace if key == "u" else self._external) or {}).items():
            v[j * d:(j + 1) * d] = vec
        return v

    def _sparse(self, key):
        """Build (once) the reference's sparse dict view of a dense result."""
        attr = {"u": "_displace", "ext": "_external", "axial": "_internal"}[key]
        cur = getattr(self, attr)
        if cur is None and self._dense is not None:
            v = self._dense[key]
            if key == "axial":
                cur = {int(m): float(v[m]) for m in np.nonzero(~(np.abs(v) < ZERO_EPS))[0]}
            else:
                rows = v.reshape(-1, self._dim)
                cur = {int(j): rows[j].copy() for j in np.nonzero(~(np.abs(rows) < ZERO_EPS).all(axis=1))[0]}
            setattr(self, attr, cur)
        return cur

    def __repr__(self):
        bar = "-" * 30

        def block(title, value, solved_only=False):
            body = pformat(value) if (self._solved or not solved_only) else "(Not Solved)"
            return f"{bar}\n{title}\n{bar}\n{body}\n\n"

        return (object.__repr__(self) + "\n" + block("Joints :", self._joints) + block("Forces :", self._forces) +
                block("Members :", self._members) + block("Displaces:", self._sparse("u"), True) +
                block("Internals:", self._sparse("axial"), True) + block("Externals:", self._sparse("ext"), True))

    # ------------------------------------------------------------------ sizes / status
    dim = property(lambda self: self._dim)
    nJoint = property(lambda self: len(self._joints))
    nMember = property(lambda self: len(self._members))
    nForce = property(lambda self: len(self._forces))
    isSolved = property(lambda self: self._solved)

    @property
    def nSupport(self):
        return sum(1 for _, s in self._joints.values() if s != SupportType.NO)

    @property
    def nResistance(self):
        return sum(SupportType.GetResistanceNumber(s, self._dim) for _, s in self._joints.values())

    @property
    def isStable(self):
        n_res = self.nResistance
        enough = self.nMember + n_res >= self.nJoint * self._dim
        return enough if self._dim == 2 else (n_res >= 6 and enough)

    @property
    def weight(self):
        return sum(member.weight for _, _, member in self._members.values())

    # ------------------------------------------------------------------ builders / setters
    def AddNewJoint(self, vector, supportType=SupportType.NO):
        self._joints[len(self._joints)] = (tuple(float(vector[i]) for i in range(self._dim)), supportType)
        self._topology_changed()

    def AddExternalForce(self, jointID, vector):
        if jointID not in self._joints:
            raise InvaildJointError(f"No such joint [{jointID}], can't add force on it.")
        if not IsZeroVector(vector):
            self._forces[jointID] = tuple(float(vector[i]) for i in range(self._dim))
            self._buckling = None                   # (the buckling factors are those of the loads)

    def AddNewMember(self, jointID0, jointID1, memberType):
        member = Member(self._joints[jointID0][0], self._joints[jointID1][0], self._dim, memberType.Copy())
        self._members[len(self._members)] = (jointID0, jointID1, member)
        self._topology_changed()

    def SetJointPosition(self, jointID, position):
        self._joints[jointID] = (position, self._joints[jointID][1])
        self._modes = None
        self._buckling = None
        for j0, j1, member in self._members.values():
            if j0 == jointID: member.SetPosition(0, position)
            if j1 == jointID: member.SetPosition(1, position)

    def SetJointPositions(self, jointPositionDict):
        for jointID, position in jointPositionDict.items():
            self.SetJointPosition(jointID, position)

    def SetSupportType(self, jointID, supportType):
        self._joints[jointID] = (self._joints[jointID][0], supportType)
        self._topology_changed()

    def SetSupportTypes(self, supportTypeDict):
        for jointID, supportType in supportTypeDict.items():
            self.SetSupportType(jointID, supportType)

    def SetMemberType(self, memberID, memberType):
        self._members[memberID][2].memberType = memberType
        self._modes = None
        self._buckling = None

    def SetMemberTypes(self, memberTypeDict, isCheckAllSet=False):
        if isCheckAllSet and self._members.keys() - memberTypeDict.keys():
            raise NotAllBeSetError("Didn't set member types to all members.")
        for memberID, memberType in memberTypeDict.items():
            self.SetMemberType(memberID, memberType)

    def SetMemberConnect(self, memberID, connect):
        member = self._members[memberID][2]
        member.SetPosition(0, self._joints[connect[0]][0])
        member.SetPosition(1, self._joints[connect[1]][0])
        self._members[memberID] = (connect[0], connect[1], member)
        self._topology_changed()

    def SetMemberConnects(self, memberConnectDict):
        for memberID, connect in memberConnectDict.items():
            self.SetMemberConnect(memberID, connect)

    # ------------------------------------------------------------------ getters (inputs)
    def GetJointPosition(self, jointID):
        return self._joints[jointID][0]

    def GetJointPositions(self):
        return {j: pos for j, (pos, _) in self._joints.items()}

    def GetSupportType(self, jointID):
        return self._joints[jointID][1]

    def GetSupportTypes(self):
        return {j: s for j, (_, s) in self._joints.items()}

    def GetMemberType(self, memberID):
        return self._members[memberID][2].memberType

    def GetMemberTypes(self):
        return {m: member.memberType for m, (_, _, member) in self._members.items()}

    def GetMemberConnect(self, memberID):
        j0, j1, _ = self._members[memberID]
        return j0, j1

    def GetMemberFromConnect(self, connect):
        for j0, j1, member in self._members.values():
            if j0 == connect[0] and j1 == connect[1]:
                return member

    def GetForce(self, jointID):
        return self._forces[jointID]

    def GetJoints(self, isProtect=True):
        return copy.deepcopy(self._joints) if isProtect else self._joints

    def GetMembers(self, isProtect=True):
        return copy.deepcopy(self._members) if isProtect else self._members

    def GetForces(self, isProtect=True):
        return copy.deepcopy(self._forces) if isProtect else self._forces

    def GetJointIDs(self):
        return list(self._joints)

    def GetMemberIDs(self):
        return list(self._members)

    def GetUsedMemberTypes(self):
        return {member.memberType for _, _, member in self._members.values()}

    # ------------------------------------------------------------------ getters (results)
    def GetDisplacements(self, isProtect=True):
        d = self._sparse("u")
        return copy.deepcopy(d) if isProtect else d

    def GetExternalForces(self, isProtect=True):
        d = self._sparse("ext")
        return copy.deepcopy(d) if isProtect else d

    def GetInternalForces(self, isProtect=True):
        d = self._sparse("axial")
        return copy.deepcopy(d) if isProtect else d

    def GetInternalStresses(self):
        internal = self._sparse("axial")
        if internal is None:
            return None
        return {m: force / self._members[m][2].a for m, force in internal.items()}

    def GetResistances(self):
        if not self._solved:
            return None
        external = self._sparse("ext")
        res = {}
        for j, (_, support) in self._joints.items():
            if support != SupportType.NO:
                reaction = external.get(j, np.zeros([self._dim]))
                res[j] = reaction - self._forces[j] if j in self._forces else reaction
        return res

    # ------------------------------------------------------------------ linear-system views
    def GetExternalForceVector(self):
        return self._pack()[4]

    def GetDisplacementUnknownMask(self):
        """bool[N], True where the displacement is unknown -- from the plan's bit-exact DOF map."""
        free_idx, _, _ = self._get_plan().maps()
        mask = np.zeros(self.nJoint * self._dim, dtype=bool)
        mask[free_idx] = True
        return mask

    def GetKMatrix(self):
        """Dense N x N stiffness matrix (inspection helper only: Solve() assembles on the GPU)."""
        xyz, _, conn, aed, _ = self._pack()
        d, N = self._dim, self.nJoint * self._dim
        K = np.zeros((N, N))
        for m, (j0, j1, member) in self._members.items():
            dofs = [j0 * d + i for i in range(d)] + [j1 * d + i for i in range(d)]
            K[np.ix_(dofs, dofs)] += member.matK
        return K

    # ------------------------------------------------------------------ the solve
    def Solve(self):
        """Direct stiffness method, K u = f, on the GPU (batch of one)."""
        if not self.isStable:
            raise TrussNotStableError("The truss is not stable !")
        xyz, support, conn, aed, force = self._pack()
        plan = self._get_plan(support, conn)
        out = plan.solve_host(1, xyz, force, aed=aed, want=("u", "ext", "axial"))
        raise_for_info(int(out["info"][0]))
        self._set_dense_results(out["u"][0], out["ext"][0], out["axial"][0])

    # ------------------------------------------------------------------ modal analysis
    def SolveModes(self, nMode=None, isConsistentMass=False, jointMasses=None):
        """Free vibration K_ff phi = lambda M_ff phi on the GPU (tb_modes, batch of one): the ``nMode`` lowest eigenpairs
        (None = all).  Member mass is (a L) density in the caller's units (divide a weight density by g first); lumped
        mass puts half of it on every axis of both end joints, ``isConsistentMass`` uses the consistent bar mass matrix.
        ``jointMasses``: {jointID: mass} added on every axis of the joint.  A mechanism that passes the counting rule is
        not an error: it shows as eigenvalues ~ 0."""
        if not self.isStable:
            raise TrussNotStableError("The truss is not stable !")
        xyz, support, conn, aed, _ = self._pack()
        plan = self._get_plan(support, conn)
        jm = None
        if jointMasses:
            jm = np.zeros(self.nJoint)
            for j, mass in jointMasses.items():
                if j not in self._joints:
                    raise InvaildJointError(f"No such joint [{j}], can't add a mass on it.")
                jm[j] = float(mass)
        out = plan.modes_host(1, xyz, aed=aed, n_modes=nMode, consistent=isConsistentMass, joint_mass=jm)
        raise_for_modes_info(int(out["info"][0]))
        self._modes = {"eigval": out["eigval"][0].copy(), "modes": out["modes"][0].copy()}

    def _modes_or_raise(self):
        if self._modes is None:
            raise TrussNotSolvedError("Haven't done modal analysis yet (SolveModes).")
        return self._modes

    def GetEigenvalues(self):
        """lambda = omega^2 of the solved modes, ascending (numpy array)."""
        return self._modes_or_raise()["eigval"].copy()

    def GetNaturalFrequencies(self):
        """Natural frequencies omega / (2 pi) of the solved modes, ascending (numpy array)."""
        return np.sqrt(np.maximum(self._modes_or_raise()["eigval"], 0.0)) / (2.0 * np.pi)

    def GetModeShapes(self):
        """One dict per mode, {jointID: displacement vector} over every joint (zero at supported DOFs), in the style of
        GetDisplacements; M-normalised, the component of largest magnitude positive."""
        modes = self._modes_or_raise()["modes"]
        d = self._dim
        return [{j: modes[k, j * d:(j + 1) * d].copy() for j in range(self.nJoint)} for k in range(modes.shape[0])]

    # ------------------------------------------------------------------ linear buckling
    def SolveBuckling(self, nMode=None):
        """Linear buckling under the current loads on the GPU: the static solve (as ``Solve``, raising as it does), then
        K_ff phi = lambda (-K_G) phi with the geometric stiffness of its member forces (tb_buckling, batch of one).  The
        ``nMode`` lowest load factors (None = one per free DOF): the loads times ``GetBucklingFactors()[0]`` make the
        truss unstable.  Modes no positive multiple of the loads reaches get an ``inf`` factor (e.g. every mode of a truss
        without compressed members).  The static results are not stored (call ``Solve`` for those)."""
        if not self.isStable:
            raise TrussNotStableError("The truss is not stable !")
        xyz, support, conn, aed, force = self._pack()
        plan = self._get_plan(support, conn)
        out = plan.solve_host(1, xyz, force, aed=aed, want=("axial",))
        raise_for_info(int(out["info"][0]))
        res = plan.buckling_host(1, xyz, out["axial"][0], aed=aed, n_modes=nMode)
        raise_for_modes_info(int(res["info"][0]))
        self._buckling = {"factor": res["factor"][0].copy(), "modes": res["modes"][0].copy()}

    def _buckling_or_raise(self):
        if self._buckling is None:
            raise TrussNotSolvedError("Haven't done buckling analysis yet (SolveBuckling).")
        return self._buckling

    def GetBucklingFactors(self):
        """Load factors of the solved buckling modes, ascending (numpy array; inf for modes no positive multiple of the
        loads reaches).  The first one is the critical load factor."""
        return self._buckling_or_raise()["factor"].copy()

    def GetBucklingModes(self):
        """One dict per buckling mode, {jointID: displacement vector} over every joint (zero at supported DOFs), in the
        style of GetModeShapes; K-normalised (phi^T K_ff phi = 1), the component of largest magnitude positive, all zero
        for a mode with an inf factor."""
        modes = self._buckling_or_raise()["modes"]
        d = self._dim
        return [{j: modes[k, j * d:(j + 1) * d].copy() for j in range(self.nJoint)} for k in range(modes.shape[0])]

    # ------------------------------------------------------------------ JSON
    def Serialize(self):
        data = {
            "joint": [[list(pos), SupportType.GetFromType(s)] for pos, s in (self._joints[j] for j in range(self.nJoint))],
            "force": [[j, list(vec)] for j, vec in self._forces.items()],
            "member": [[[j0, j1], member.memberType.Serialize()]
                       for j0, j1, member in (self._members[m] for m in range(self.nMember))],
        }
        if self._solved:
            data["displace"] = [[j, list(v)] for j, v in self._sparse("u").items()]
            data["external"] = [[j, list(v)] for j, v in self._sparse("ext").items()]
            data["internal"] = [[m, float(f)] for m, f in self._sparse("axial").items()]
            data["weight"] = self.weight
        return data

    def LoadFromJSON(self, path=None, isOutputFile=False, data=None):
        if data is None:
            with open(path, "r", encoding="utf-8") as f:
                data = json.load(f)
        for vector, support in data["joint"]:
            self.AddNewJoint(vector, SupportType.GetFromString(support))
        for jointID, vector in data["force"]:
            self.AddExternalForce(jointID, vector)
        for (j0, j1), memberType in data["member"]:
            self.AddNewMember(j0, j1, MemberType(*memberType))
        if isOutputFile:
            self._dense = None
            self._displace = {j: np.array(v) for j, v in data["displace"]}
            self._external = {j: np.array(v) for j, v in data["external"]}
            self._internal = {m: float(f) for m, f in data["internal"]}
            self._solved = True
        return self

    def DumpIntoJSON(self, path):
        with open(path, "w", encoding="utf-8") as f:
            json.dump(self.Serialize(), f, ensure_ascii=False)

    # ------------------------------------------------------------------ allowable-limit checks
    def _limit_check(self, values, limit, isGetSumViolation, isGetSumNonViolation):
        over = {k: v - limit for k, v in values.items() if v > limit}
        if isGetSumViolation:
            violation = sum(over.values())
            ok = IsZero(violation)
        else:
            violation, ok = over, len(over) == 0
        if isGetSumNonViolation:
            return ok, violation, sum(limit - v for v in values.values() if v <= limit)
        return ok, violation

    def IsInternalStressAllowed(self, limit, isGetSumViolation=False, isGetSumNonViolation=False):
        if not self._solved:
            raise TrussNotSolvedError("Haven't done structural analysis yet.")
        stress = {m: abs(f) / self._members[m][2].a for m, f in self._sparse("axial").items()}
        return self._limit_check(stress, limit, isGetSumViolation, isGetSumNonViolation)

    def IsDisplacementAllowed(self, limit, isGetSumViolation=False, isGetSumNonViolation=False):
        if not self._solved:
            raise TrussNotSolvedError("Haven't done structural analysis yet.")
        norms = {j: GetLength(v) for j, v in self._sparse("u").items()}
        return self._limit_check(norms, limit, isGetSumViolation, isGetSumNonViolation)

    def Copy(self):
        return Truss(self._dim).LoadFromJSON(data=self.Serialize(), isOutputFile=self._solved)
