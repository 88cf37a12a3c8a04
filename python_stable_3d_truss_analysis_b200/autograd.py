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
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib

__all__ = ["solve", "solve_ragged"]


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

        def per_input(g, x):                      # a shared (unbatched) input gets the sum over the batch
            if g is None:
                return None
            return g.reshape(x.shape) if x.dim() == g.dim() else g.sum(0)

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
    for k, t in list(base.items()) + [("xyz", xyz), ("aed", aed), ("force", force)]:   # (dtypes and shapes first)
        if not t.is_cuda or t.device != xyz.device:
            raise TypeError(f"{k} must be a CUDA tensor on the device of xyz")
    xyz, aed, force = xyz.contiguous(), aed.contiguous(), force.contiguous()
    jo, mo = base["joint_off"], base["member_off"]
    if (max_joint is None or max_member is None) and jo.shape[0] > 1:      # one device-to-host read for both passes
        mj, mm = torch.stack([(jo[1:] - jo[:-1]).max(), (mo[1:] - mo[:-1]).max()]).tolist()
        max_joint = mj if max_joint is None else max_joint
        max_member = mm if max_member is None else max_member
    with torch.cuda.device(xyz.device):
        u, ext, axial, weight, info = _SolveRagged.apply(xyz, aed, force, base["joint_off"], base["member_off"], base["support"],
                                                         base["conn"], dim, max_joint, max_member)
    return {"u": u, "ext": ext, "axial": axial, "weight": weight, "info": info}
