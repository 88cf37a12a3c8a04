"""Differentiable truss solve for ``torch.autograd``.

``solve(truss, xyz, aed, force)`` runs ``Truss.Solve()`` (truss.py:329-364) for a batch of systems on the GPU and returns
displacements, loads with reactions, member forces and weights that backpropagate to the joint coordinates (shape), the
member properties (sizing) and the loads.  The backward pass is one adjoint solve with the same stiffness matrix
(``tb_adjoint``, DESIGN.md section 9), so a gradient costs about one more solve.

Example -- compliance gradient of bar-72 with respect to the member areas::

    aed = torch.tensor(aed0, dtype=torch.float64, device="cuda", requires_grad=True)
    f = torch.tensor(f0, dtype=torch.float64, device="cuda")
    out = autograd.solve(truss, aed=aed, force=f)
    (f * out["u"]).sum().backward()                   # compliance C = f.u
    dC_dA = aed.grad[:, 0]

``solve_ragged(packed, xyz, aed, force)`` does the same for a ragged batch -- every truss with its own topology, packed
back to back as ``gencube_device`` / ``augment_and_solve_device`` return them (``tb_adjoint_ragged``).

``modes(truss, xyz, aed, joint_mass)`` runs the modal analysis (``tb_modes``, DESIGN.md section 11) and returns eigenvalues
that backpropagate to the joint coordinates, the member properties and the joint masses (``tb_modes_adjoint``: one pass
over the members, nothing solved).  Example -- a frequency penalty for sizing, symmetric in the eigenvalues::

    out = autograd.modes(truss, aed=aed, n_modes=6)
    penalty = torch.relu(lam_min - out["eigval"]).pow(2).sum()
    penalty.backward()                                # aed.grad

``modes_ragged(packed, xyz, aed, joint_mass)`` does the same for a ragged batch (``tb_modes_ragged`` /
``tb_modes_adjoint_ragged``).

``buckling(truss, xyz, aed, force=force)`` runs the static solve and then linear buckling (``tb_buckling``, DESIGN.md
section 12) under its member forces, and returns load factors that backpropagate to the joint coordinates, the member
properties and the loads (``tb_buckling_adjoint``, then ``tb_adjoint`` for the member forces' share).  Example -- a
weight-minimising sizing step with the stability constraint "critical load factor >= 1.5" as a penalty::

    aed = torch.cat([area[:, None], aed0[:, 1:]], 1)  # area: the design variables, requires_grad=True
    weight = autograd.solve(truss, aed=aed)["weight"]
    factor = autograd.buckling(truss, aed=aed, n_modes=6)["factor"]
    loss = weight + c * torch.relu(1.5 - factor[..., 0])
    loss.backward()                                   # area.grad
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib

__all__ = ["solve", "solve_ragged", "modes", "modes_ragged", "buckling"]


def per_input(g, x):
    """The gradient of input ``x`` from per-system gradients ``g``: a shared (unbatched) input gets the sum over the
    batch."""
    if g is None:
        return None
    return g.reshape(x.shape) if x.dim() == g.dim() else g.sum(0)


class _Solve(torch.autograd.Function):
    @staticmethod
    def forward(ctx, xyz, aed, force, plan, B, shared_factor):
        f64 = dict(dtype=torch.float64, device=xyz.device)
        out = {"u": torch.empty(B, plan.N, **f64), "ext": torch.empty(B, plan.N, **f64),
               "axial": torch.empty(B, plan.M, **f64), "weight": torch.empty(B, **f64),
               "info": torch.empty(B, dtype=torch.int32, device=xyz.device)}
        plan.solve_device(B, xyz, force, aed=aed, out=out, shared_factor=shared_factor)
        ctx.save_for_backward(xyz, aed, force, out["u"])
        ctx.plan, ctx.B, ctx.shared_factor = plan, B, shared_factor
        ctx.mark_non_differentiable(out["info"])
        ctx.set_materialize_grads(False)          # an output without a cotangent is passed to the library as NULL
        return out["u"], out["ext"], out["axial"], out["weight"], out["info"]

    @staticmethod
    def backward(ctx, g_u, g_ext, g_axial, g_w, _g_info):
        xyz, aed, force, u = ctx.saved_tensors
        plan, B = ctx.plan, ctx.B
        f64 = dict(dtype=torch.float64, device=xyz.device)
        grads = {k: None if g is None else g.contiguous()
                 for k, g in (("u", g_u), ("ext", g_ext), ("axial", g_axial), ("weight", g_w))}
        need_x, need_a, need_f = ctx.needs_input_grad[:3]
        res = {"joint_xyz": torch.empty(B, plan.nJ, plan.dim, **f64) if need_x else None,
               "member_aed": torch.empty(B, plan.M, 3, **f64),
               "force": torch.empty(B, plan.N, **f64) if need_f else None}
        plan.adjoint_device(B, xyz, force, aed, u, grads, res, shared_factor=ctx.shared_factor)
        return (per_input(res["joint_xyz"], xyz), per_input(res["member_aed"], aed) if need_a else None,
                per_input(res["force"], force), None, None, None)


def _input(t, default, row_shape, device, name):
    """(tensor, batch size or None) for an input given as [*row_shape], [B, *row_shape] or None (the truss's own)."""
    if t is None:
        return torch.as_tensor(np.ascontiguousarray(default, dtype=np.float64).reshape(row_shape), device=device), None
    if not isinstance(t, torch.Tensor) or t.dtype != torch.float64 or not t.is_cuda:
        raise TypeError(f"{name} must be a float64 CUDA tensor")
    if tuple(t.shape) == row_shape:
        return t.contiguous(), None
    if t.dim() == len(row_shape) + 1 and tuple(t.shape[1:]) == row_shape:
        return t.contiguous(), int(t.shape[0])
    raise ValueError(f"{name} must have shape {list(row_shape)} or [B, {', '.join(map(str, row_shape))}], "
                     f"not {list(t.shape)}")


def solve(truss, xyz=None, aed=None, force=None, shared_factor=False):
    """``Truss.Solve()`` for a uniform batch, differentiable with respect to ``xyz``, ``aed`` and ``force``.

    Inputs are float64 CUDA tensors: ``xyz`` [nJ, d] joint positions, ``aed`` [M, 3] (a, e, density) per member,
    ``force`` [N] dense loads (index joint * d + axis); each either unbatched (shared by every system) or with a
    leading batch dimension B.  ``None`` means the truss's own values, held constant.  ``shared_factor``: the systems
    are load cases of one truss (only ``force`` batched) and share one factorisation on the band path.

    Returns ``{"u": [B, N], "ext": [B, N], "axial": [B, M], "weight": [B], "info": [B] int32}`` (without the batch
    dimension when no input has one).  ``info`` is the per-system status of ``include/truss_b200.h`` and is not
    differentiable; a failed system has zero outputs and zero gradients."""
    pxyz, psup, pconn, paed, pforce = truss._pack()
    plan = truss._get_plan(psup, pconn)
    given = [t for t in (xyz, aed, force) if isinstance(t, torch.Tensor)]
    device = given[0].device if given else torch.device("cuda", torch.cuda.current_device())
    xyz, bx = _input(xyz, pxyz, (plan.nJ, plan.dim), device, "xyz")
    aed, ba = _input(aed, paed, (plan.M, 3), device, "aed")
    force, bf = _input(force, pforce, (plan.N,), device, "force")
    sizes = {b for b in (bx, ba, bf) if b is not None}
    if len(sizes) > 1:
        raise ValueError(f"batched inputs disagree on the batch size: {sorted(sizes)}")
    B = sizes.pop() if sizes else 1
    with torch.cuda.device(device):
        u, ext, axial, weight, info = _Solve.apply(xyz, aed, force, plan, B, bool(shared_factor))
    out = {"u": u, "ext": ext, "axial": axial, "weight": weight, "info": info}
    if bx is None and ba is None and bf is None:
        out = {k: v[0] for k, v in out.items()}
    return out


class _SolveRagged(torch.autograd.Function):
    @staticmethod
    def forward(ctx, xyz, aed, force, joint_off, member_off, support, conn, dim, maxj, maxm):
        p = dict(joint_off=joint_off, member_off=member_off, support=support, conn=conn, xyz=xyz, aed=aed, force=force)
        out = _lib.solve_ragged_device(dim, p, max_joint=maxj, max_member=maxm)
        # (the topology tensors too: the version counter then refuses a backward after an in-place change to them)
        ctx.save_for_backward(xyz, aed, force, out["u"], joint_off, member_off, support, conn)
        ctx.dim, ctx.maxj, ctx.maxm = dim, maxj, maxm
        ctx.mark_non_differentiable(out["info"])
        ctx.set_materialize_grads(False)          # an output without a cotangent is passed to the library as NULL
        return out["u"], out["ext"], out["axial"], out["weight"], out["info"]

    @staticmethod
    def backward(ctx, g_u, g_ext, g_axial, g_w, _g_info):
        xyz, aed, force, u, joint_off, member_off, support, conn = ctx.saved_tensors
        grads = {k: None if g is None else g.contiguous()
                 for k, g in (("u", g_u), ("ext", g_ext), ("axial", g_axial), ("weight", g_w))}
        need_x, _, need_f = ctx.needs_input_grad[:3]
        res = {"joint_xyz": torch.empty_like(xyz) if need_x else None, "member_aed": torch.empty_like(aed),
               "force": torch.empty_like(force) if need_f else None,
               "info": torch.empty(joint_off.shape[0] - 1, dtype=torch.int32, device=u.device)}
        p = dict(joint_off=joint_off, member_off=member_off, support=support, conn=conn, xyz=xyz, aed=aed, force=force)
        _lib.adjoint_ragged_device(ctx.dim, p, u, grads, res, max_joint=ctx.maxj, max_member=ctx.maxm)
        return (res["joint_xyz"], res["member_aed"] if ctx.needs_input_grad[1] else None, res["force"]) + (None,) * 7


def _packed_input(t, default, shapes, name):
    """``t`` (the packed default when None) after checking that it is a float64 tensor of one of ``shapes``."""
    if t is None:
        t = default
    if not isinstance(t, torch.Tensor) or t.dtype != torch.float64:
        raise TypeError(f"{name} must be a float64 CUDA tensor")
    if tuple(t.shape) not in shapes:
        raise ValueError(f"{name} must have shape {' or '.join(str(list(s)) for s in shapes)}, not {list(t.shape)}")
    return t


def _refuse_beyond_fused(dim, joint_off, max_joint, max_member):
    """Reverse mode exists for the fused kernels' trusses only: a batch beyond them (which the forward would solve on the
    envelope kernel) is refused before any launch."""
    if joint_off.shape[0] > 1 and not _lib.small_path_fits(dim, max_joint, max_member):
        raise _lib.TrussLibError(_lib.TB_ERR_TOO_LARGE, "no reverse mode for a ragged batch beyond the fused kernels")


def solve_ragged(packed, xyz=None, aed=None, force=None, max_joint=None, max_member=None):
    """``Truss.Solve()`` for a ragged batch (every truss its own topology), differentiable with respect to ``xyz``,
    ``aed`` and ``force``.

    ``packed`` is a dict of CUDA tensors in the layout of ``tb_ragged_in``: ``joint_off`` / ``member_off`` [B+1] int64,
    ``support`` [sum nJ] uint8, ``conn`` [2 sum M] int32 (local joint ids) and optionally ``xyz`` / ``aed`` / ``force``
    -- what ``_lib.gencube_device`` and ``_lib.augment_and_solve_device`` return (a ``PackedDataset``'s arrays moved to
    the device work too).  ``xyz`` [sum nJ, d] or [d sum nJ], ``aed`` [sum M, 3] or [3 sum M] and ``force`` [d sum nJ] are
    float64 CUDA tensors; None means the packed value, held constant.  ``max_joint`` / ``max_member`` size the kernels;
    None reads them from the offsets (one device-to-host copy).

    Returns ``{"u": [d sum nJ], "ext": [d sum nJ], "axial": [sum M], "weight": [B], "info": [B] int32}`` in the packed
    layout.  ``info`` is the per-truss status of ``include/truss_b200.h`` and is not differentiable; a failed truss has
    zero outputs and zero gradients.  Every input row belongs to one truss, so the gradients need no batch reduction."""
    for k, dt in (("joint_off", torch.int64), ("member_off", torch.int64), ("support", torch.uint8), ("conn", torch.int32)):
        t = packed.get(k)
        if not isinstance(t, torch.Tensor) or t.dtype != dt or t.dim() != 1:
            raise TypeError(f"packed[{k!r}] must be a 1-D {dt} CUDA tensor")
    SJ, SM = int(packed["support"].numel()), int(packed["conn"].numel()) // 2
    src = xyz if xyz is not None else packed.get("xyz")
    if isinstance(src, torch.Tensor) and src.dim() == 2:
        dim = int(src.shape[1])
    elif isinstance(src, torch.Tensor) and SJ > 0 and src.numel() % SJ == 0:
        dim = src.numel() // SJ
    else:
        raise ValueError("xyz must have shape [sum nJ, d] or [d * sum nJ] with d = 2 or 3")
    if dim not in (2, 3):
        raise ValueError(f"xyz must have d = 2 or 3 columns, not {dim}")
    xyz = _packed_input(xyz, packed.get("xyz"), [(SJ, dim), (SJ * dim,)], "xyz")
    aed = _packed_input(aed, packed.get("aed"), [(SM, 3), (SM * 3,)], "aed")
    force = _packed_input(force, packed.get("force"), [(SJ * dim,)], "force")
    base = {k: packed[k] for k in ("joint_off", "member_off", "support", "conn")}
    if max_joint is not None and max_member is not None:                 # (sizes known: refused before anything else)
        _refuse_beyond_fused(dim, base["joint_off"], max_joint, max_member)
    for k, t in list(base.items()) + [("xyz", xyz), ("aed", aed), ("force", force)]:   # (dtypes and shapes first)
        if not t.is_cuda or t.device != xyz.device:
            raise TypeError(f"{k} must be a CUDA tensor on the device of xyz")
    xyz, aed, force = xyz.contiguous(), aed.contiguous(), force.contiguous()
    jo, mo = base["joint_off"], base["member_off"]
    if (max_joint is None or max_member is None) and jo.shape[0] > 1:      # one device-to-host read for both passes
        mj, mm = torch.stack([(jo[1:] - jo[:-1]).max(), (mo[1:] - mo[:-1]).max()]).tolist()
        max_joint = mj if max_joint is None else max_joint
        max_member = mm if max_member is None else max_member
    _refuse_beyond_fused(dim, jo, max_joint, max_member)
    with torch.cuda.device(xyz.device):
        u, ext, axial, weight, info = _SolveRagged.apply(xyz, aed, force, base["joint_off"], base["member_off"], base["support"],
                                                         base["conn"], dim, max_joint, max_member)
    return {"u": u, "ext": ext, "axial": axial, "weight": weight, "info": info}


class _Modes(torch.autograd.Function):
    @staticmethod
    def forward(ctx, xyz, aed, joint_mass, plan, B, n_modes, consistent):
        out = {"modes": torch.empty(B, n_modes, plan.N, dtype=torch.float64, device=xyz.device)}   # (the backward needs them)
        plan.modes_device(B, xyz, aed=aed, n_modes=n_modes, consistent=consistent, joint_mass=joint_mass, out=out)
        ctx.save_for_backward(xyz, aed, joint_mass, out["eigval"], out["modes"], out["info"])
        ctx.plan, ctx.B, ctx.n_modes, ctx.consistent = plan, B, n_modes, consistent
        ctx.mark_non_differentiable(out["modes"], out["info"])
        ctx.set_materialize_grads(False)
        return out["eigval"], out["modes"], out["info"]

    @staticmethod
    def backward(ctx, g_eigval, _g_modes, _g_info):
        if g_eigval is None:
            return (None,) * 7
        xyz, aed, joint_mass, eigval, modes_, info = ctx.saved_tensors
        plan, B = ctx.plan, ctx.B
        f64 = dict(dtype=torch.float64, device=xyz.device)
        need_x, need_a, need_m = ctx.needs_input_grad[:3]
        res = {"joint_xyz": torch.empty(B, plan.nJ, plan.dim, **f64) if need_x else None,
               "member_aed": torch.empty(B, plan.M, 3, **f64) if need_a else None,
               "joint_mass": torch.empty(B, plan.nJ, **f64) if need_m else None}
        fwd = {"eigval": eigval, "modes": modes_, "info": info}
        plan.modes_adjoint_device(B, xyz, aed, fwd, g_eigval.contiguous(), res, n_modes=ctx.n_modes, consistent=ctx.consistent)
        return (per_input(res["joint_xyz"], xyz), per_input(res["member_aed"], aed),
                per_input(res["joint_mass"], joint_mass) if need_m else None, None, None, None, None)


def modes(truss, xyz=None, aed=None, joint_mass=None, n_modes=None, consistent=False):
    """Modal analysis (``Truss.SolveModes``) for a uniform batch, with eigenvalues differentiable with respect to
    ``xyz``, ``aed`` and ``joint_mass``.

    Inputs are float64 CUDA tensors: ``xyz`` [nJ, d] joint positions, ``aed`` [M, 3] (a, e, density) per member and
    ``joint_mass`` [nJ] non-structural mass per joint; each either unbatched (shared by every system) or with a leading
    batch dimension B.  ``xyz`` / ``aed`` None mean the truss's own values, held constant; ``joint_mass`` None means no
    non-structural mass.  ``n_modes`` (None = all n free DOFs) lowest modes; ``consistent`` selects the consistent mass
    matrix instead of the lumped one.

    Returns ``{"eigval": [B, k], "modes": [B, k, N], "info": [B] int32}`` (without the batch dimension when no input has
    one): lambda = omega^2 ascending, M-normalised mode shapes (0 at supported DOFs) and the per-system status of
    ``include/truss_b200.h``.  Only ``eigval`` is differentiable (dlambda/dp = phi^T (dK/dp - lambda dM/dp) phi); a
    failed system has zero outputs and zero gradients.

    Repeated eigenvalues (bar-72 and bar-120 have an exactly repeated lowest pair): a single eigenvalue of a cluster is
    not differentiable, only functions symmetric in the cluster's eigenvalues are.  A loss that treats every mode alike
    -- ``relu(lam_min - eigval).pow(2).sum()``, ``(1 / eigval).sum()`` -- sends equal cotangents to a cluster and gets
    its exact gradient, whatever basis of the cluster the forward returned.  A loss that singles out one eigenvalue of a
    cluster (``eigval[..., 0]`` on bar-72) gets a basis-dependent directional value; so does any loss when ``n_modes``
    cuts a cluster in two.  Ask for enough modes to keep the clusters you use whole."""
    pxyz, psup, pconn, paed, _ = truss._pack()
    plan = truss._get_plan(psup, pconn)
    given = [t for t in (xyz, aed, joint_mass) if isinstance(t, torch.Tensor)]
    device = given[0].device if given else torch.device("cuda", torch.cuda.current_device())
    xyz, bx = _input(xyz, pxyz, (plan.nJ, plan.dim), device, "xyz")
    aed, ba = _input(aed, paed, (plan.M, 3), device, "aed")
    bm = None
    if joint_mass is not None:
        joint_mass, bm = _input(joint_mass, None, (plan.nJ,), device, "joint_mass")
    for name, t in (("xyz", xyz), ("aed", aed), ("joint_mass", joint_mass)):
        if t is not None and t.device != device:
            raise TypeError(f"{name} must be on the device of the other inputs ({device})")
    sizes = {b for b in (bx, ba, bm) if b is not None}
    if len(sizes) > 1:
        raise ValueError(f"batched inputs disagree on the batch size: {sorted(sizes)}")
    B = sizes.pop() if sizes else 1
    k = plan.n if n_modes is None else int(n_modes)
    with torch.cuda.device(device):
        eigval, shapes, info = _Modes.apply(xyz, aed, joint_mass, plan, B, k, bool(consistent))
    out = {"eigval": eigval, "modes": shapes, "info": info}
    if bx is None and ba is None and bm is None:
        out = {key: v[0] for key, v in out.items()}
    return out


class _Buckling(torch.autograd.Function):
    @staticmethod
    def forward(ctx, xyz, aed, axial, plan, B, n_modes):
        out = {"modes": torch.empty(B, n_modes, plan.N, dtype=torch.float64, device=xyz.device)}   # (the backward needs them)
        plan.buckling_device(B, xyz, axial, aed=aed, n_modes=n_modes, out=out)
        ctx.save_for_backward(xyz, aed, axial, out["factor"], out["modes"], out["info"])
        ctx.plan, ctx.B, ctx.n_modes = plan, B, n_modes
        ctx.mark_non_differentiable(out["modes"], out["info"])
        ctx.set_materialize_grads(False)
        return out["factor"], out["modes"], out["info"]

    @staticmethod
    def backward(ctx, g_factor, _g_modes, _g_info):
        if g_factor is None:
            return (None,) * 6
        xyz, aed, axial, factor, modes_, info = ctx.saved_tensors
        plan, B = ctx.plan, ctx.B
        f64 = dict(dtype=torch.float64, device=xyz.device)
        need_x, need_a, need_n = ctx.needs_input_grad[:3]
        res = {"joint_xyz": torch.empty(B, plan.nJ, plan.dim, **f64) if need_x else None,
               "member_aed": torch.empty(B, plan.M, 3, **f64) if need_a else None,
               "axial": torch.empty(B, plan.M, **f64) if need_n else None}
        fwd = {"factor": factor, "modes": modes_, "info": info}
        plan.buckling_adjoint_device(B, xyz, aed, axial, fwd, g_factor.contiguous(), res, n_modes=ctx.n_modes)
        return (per_input(res["joint_xyz"], xyz), per_input(res["member_aed"], aed), per_input(res["axial"], axial),
                None, None, None)


def buckling(truss, xyz=None, aed=None, axial=None, force=None, n_modes=None):
    """Linear buckling (``Truss.SolveBuckling``) for a uniform batch, with load factors differentiable with respect to
    ``xyz``, ``aed`` and the loads or the member forces.

    Inputs are float64 CUDA tensors: ``xyz`` [nJ, d] joint positions, ``aed`` [M, 3] (a, e, density) per member, and
    either ``axial`` [M], the member forces N of the reference state (tension positive), or ``force`` [N], dense loads
    (index joint * d + axis); each either unbatched (shared by every system) or with a leading batch dimension B.
    ``xyz`` / ``aed`` / ``force`` None mean the truss's own values, held constant.  With ``axial`` None the member forces
    come from ``solve(truss, xyz, aed, force)``, so the gradients also flow through the static solve (one adjoint solve)
    and reach the loads.  ``n_modes`` (None = all n free DOFs) lowest factors.

    Returns ``{"factor": [B, k], "modes": [B, k, N], "info": [B] int32, "axial": [B, M]}`` (without the batch dimension
    when no input has one): the load factors ascending (+inf for modes no positive multiple of N reaches), the
    K-normalised buckling modes (0 at supported DOFs), the per-system status of ``include/truss_b200.h`` and the member
    forces used.  Only ``factor`` (and ``axial``, when it comes from the solve) is differentiable
    (dlambda/dp = lambda phi^T dK/dp phi + lambda^2 phi^T dK_G/dp phi); a failed system has zero outputs and zero
    gradients, and a factor at +inf has zero gradient whatever its cotangent.

    Repeated factors (symmetric structures such as a column braced alike in two directions have exactly repeated
    critical pairs): a single factor of a cluster is not differentiable, only functions symmetric in the cluster's
    factors are.  A loss that treats every factor alike -- ``relu(1.5 - factor).sum()`` -- sends equal cotangents to a
    cluster and gets its exact gradient, whatever basis of the cluster the forward returned.  A loss that singles out
    one factor of a cluster (``factor[..., 0]`` when the lowest factor is a pair) gets a basis-dependent directional
    value; so does any loss when ``n_modes`` cuts a cluster in two.  Ask for enough modes to keep the clusters you use
    whole."""
    if axial is not None and force is not None:
        raise ValueError("give the member forces (axial) or the loads (force), not both")
    pxyz, psup, pconn, paed, pforce = truss._pack()
    plan = truss._get_plan(psup, pconn)
    given = [t for t in (xyz, aed, axial, force) if isinstance(t, torch.Tensor)]
    device = given[0].device if given else torch.device("cuda", torch.cuda.current_device())
    xyz, bx = _input(xyz, pxyz, (plan.nJ, plan.dim), device, "xyz")
    aed, ba = _input(aed, paed, (plan.M, 3), device, "aed")
    if axial is not None:
        axial, bl = _input(axial, None, (plan.M,), device, "axial")
    else:
        force, bl = _input(force, pforce, (plan.N,), device, "force")
    for name, t in (("xyz", xyz), ("aed", aed), ("axial", axial), ("force", force)):
        if t is not None and t.device != device:
            raise TypeError(f"{name} must be on the device of the other inputs ({device})")
    sizes = {b for b in (bx, ba, bl) if b is not None}
    if len(sizes) > 1:
        raise ValueError(f"batched inputs disagree on the batch size: {sorted(sizes)}")
    B = sizes.pop() if sizes else 1
    k = plan.n if n_modes is None else int(n_modes)
    with torch.cuda.device(device):
        if axial is None:
            axial = solve(truss, xyz, aed, force)["axial"]
        factor, shapes, info = _Buckling.apply(xyz, aed, axial, plan, B, k)
    out = {"factor": factor, "modes": shapes, "info": info}
    if bx is None and ba is None and bl is None:
        out = {key: v[0] for key, v in out.items()}
    out["axial"] = axial
    return out


class _ModesRagged(torch.autograd.Function):
    @staticmethod
    def forward(ctx, xyz, aed, joint_mass, joint_off, member_off, support, conn, dim, n_modes, consistent, sizes):
        p = dict(joint_off=joint_off, member_off=member_off, support=support, conn=conn, xyz=xyz, aed=aed)
        mj, mm, mf = sizes
        out = _lib.modes_ragged_device(dim, p, n_modes, consistent=consistent, joint_mass=joint_mass, max_joint=mj,
                                       max_member=mm, max_free=mf)
        ctx.save_for_backward(xyz, aed, joint_mass, out["eigval"], out["modes"], out["info"], joint_off, member_off,
                              support, conn)
        ctx.dim, ctx.consistent, ctx.sizes = dim, consistent, sizes
        ctx.mark_non_differentiable(out["modes"], out["n_free"], out["info"])
        ctx.set_materialize_grads(False)
        return out["eigval"], out["modes"], out["n_free"], out["info"]

    @staticmethod
    def backward(ctx, g_eigval, _g_modes, _g_nfree, _g_info):
        if g_eigval is None:
            return (None,) * 11
        xyz, aed, joint_mass, eigval, modes_, info, joint_off, member_off, support, conn = ctx.saved_tensors
        need_x, need_a, need_m = ctx.needs_input_grad[:3]
        res = {"joint_xyz": torch.empty_like(xyz) if need_x else None, "member_aed": torch.empty_like(aed) if need_a else None,
               "joint_mass": torch.empty_like(joint_mass) if need_m else None}
        p = dict(joint_off=joint_off, member_off=member_off, support=support, conn=conn, xyz=xyz, aed=aed)
        mj, mm, mf = ctx.sizes
        _lib.modes_adjoint_ragged_device(ctx.dim, p, {"eigval": eigval, "modes": modes_, "info": info}, g_eigval.contiguous(),
                                         res, consistent=ctx.consistent, max_joint=mj, max_member=mm, max_free=mf)
        return (res["joint_xyz"], res["member_aed"], res["joint_mass"]) + (None,) * 8


def modes_ragged(packed, xyz=None, aed=None, joint_mass=None, n_modes=6, consistent=False, max_joint=None,
                 max_member=None, max_free=None):
    """Modal analysis of a ragged batch (every truss its own topology), with eigenvalues differentiable with respect to
    ``xyz``, ``aed`` and ``joint_mass``.

    ``packed`` is a dict of CUDA tensors in the layout of ``tb_ragged_in`` (as for ``solve_ragged``; ``force`` is not
    used).  ``xyz`` [sum nJ, d] or [d sum nJ], ``aed`` [sum M, 3] or [3 sum M] and ``joint_mass`` [sum nJ] are float64
    CUDA tensors; ``xyz`` / ``aed`` None mean the packed values held constant, ``joint_mass`` None no non-structural
    mass.  ``n_modes`` lowest modes per truss; ``consistent`` selects the consistent mass matrix.  ``max_joint`` /
    ``max_member`` / ``max_free`` size the kernels; None reads them from the offsets and support codes (one
    device-to-host copy).  ``max_free`` defaults to the largest truss's free-DOF count (at least ``n_modes``).

    Returns ``{"eigval": [B, k], "modes": [k d sum nJ], "n_free": [B] int32, "info": [B] int32}``: per truss lambda =
    omega^2 ascending, its M-normalised mode shapes as the block ``[k][d nJ_b]`` starting at ``k d joint_off[b]``, its
    free-DOF count and its status (``include/truss_b200.h``).  A truss with fewer than k free DOFs gets zeros past
    ``n_free[b]``, which take no part in the gradient.  Only ``eigval`` is differentiable; a failed truss has zero outputs
    and zero gradients.

    Repeated eigenvalues: a single eigenvalue of a cluster is not differentiable, only functions symmetric in the
    cluster's eigenvalues are.  A loss that treats every mode alike -- ``relu(lam_min - eigval).pow(2).sum()``,
    ``(1 / eigval).sum()`` -- sends equal cotangents to a cluster and gets its exact gradient, whatever basis of the
    cluster the forward returned.  A loss that singles out one eigenvalue of a cluster gets a basis-dependent
    directional value; so does any loss when ``n_modes`` cuts a cluster in two.  Ask for enough modes to keep the
    clusters you use whole."""
    for k, dt in (("joint_off", torch.int64), ("member_off", torch.int64), ("support", torch.uint8), ("conn", torch.int32)):
        t = packed.get(k)
        if not isinstance(t, torch.Tensor) or t.dtype != dt or t.dim() != 1:
            raise TypeError(f"packed[{k!r}] must be a 1-D {dt} CUDA tensor")
    n_modes = int(n_modes)
    if n_modes < 1:
        raise ValueError(f"n_modes must be at least 1, not {n_modes}")
    SJ, SM = int(packed["support"].numel()), int(packed["conn"].numel()) // 2
    src = xyz if xyz is not None else packed.get("xyz")
    if isinstance(src, torch.Tensor) and src.dim() == 2:
        dim = int(src.shape[1])
    elif isinstance(src, torch.Tensor) and SJ > 0 and src.numel() % SJ == 0:
        dim = src.numel() // SJ
    else:
        raise ValueError("xyz must have shape [sum nJ, d] or [d * sum nJ] with d = 2 or 3")
    if dim not in (2, 3):
        raise ValueError(f"xyz must have d = 2 or 3 columns, not {dim}")
    xyz = _packed_input(xyz, packed.get("xyz"), [(SJ, dim), (SJ * dim,)], "xyz")
    aed = _packed_input(aed, packed.get("aed"), [(SM, 3), (SM * 3,)], "aed")
    if joint_mass is not None:
        joint_mass = _packed_input(joint_mass, None, [(SJ,)], "joint_mass")
    base = {k: packed[k] for k in ("joint_off", "member_off", "support", "conn")}
    for k, t in list(base.items()) + [("xyz", xyz), ("aed", aed), ("joint_mass", joint_mass)]:
        if t is not None and (not t.is_cuda or t.device != xyz.device):
            raise TypeError(f"{k} must be a CUDA tensor on the device of xyz")
    xyz, aed = xyz.contiguous(), aed.contiguous()
    joint_mass = joint_mass.contiguous() if joint_mass is not None else None
    with torch.cuda.device(xyz.device):
        sizes = _lib._modes_ragged_sizes(dim, base, n_modes, max_joint, max_member, max_free)
        eigval, shapes, n_free, info = _ModesRagged.apply(xyz, aed, joint_mass, base["joint_off"], base["member_off"],
                                                          base["support"], base["conn"], dim, n_modes, bool(consistent), sizes)
    return {"eigval": eigval, "modes": shapes, "n_free": n_free, "info": info}
