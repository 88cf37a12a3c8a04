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
"""
from __future__ import annotations

import numpy as np
import torch

__all__ = ["solve"]


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
