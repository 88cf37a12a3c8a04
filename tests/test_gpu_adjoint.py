"""Reverse mode of the solve on the GPU (tb_adjoint, autograd.solve) against the numpy adjoint of oracle/adjoint.py,
which tests/test_adjoint_cpu.py checks against finite differences.  Tolerance: 1e-9 norm-wise per gradient field, the
forward's parity contract."""
import json

import numpy as np
import pytest

from oracle import adjoint as adj
from oracle import truss_oracle as orc
from python_stable_3d_truss_analysis_b200 import _lib
from python_stable_3d_truss_analysis_b200.truss import Truss
from tests import helpers as H

pytestmark = pytest.mark.gpu

FIELDS = ("joint_xyz", "member_aed", "force")
PATHS = pytest.mark.parametrize("path", [0, 1, 2], ids=["fused", "tiled", "band"])


def _torch():
    import torch
    return torch


def force_path(plan, path):
    try:
        plan.set_path(path)
    except _lib.TrussLibError as exc:
        if exc.code == _lib.TB_ERR_TOO_LARGE:
            pytest.skip("system does not fit this pipeline")
        raise


def device_adjoint(plan, xyz, aed, force, grads, shared_factor=False):
    """Forward (tb_solve / tb_solve_loadcases) and reverse (tb_adjoint) on numpy inputs whose leading dimension, when
    they have one more than a single system's, is the batch.  Returns numpy dicts (forward, gradients)."""
    torch = _torch()
    dev = torch.device("cuda:0")
    td = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(dev)  # noqa: E731
    B = max(np.asarray(a).shape[0] if np.asarray(a).ndim == nd + 1 else 1
            for a, nd in ((xyz, 2), (aed, 2), (force, 1)))
    f64 = dict(dtype=torch.float64, device=dev)
    fwd = {"u": torch.empty(B, plan.N, **f64), "ext": torch.empty(B, plan.N, **f64), "axial": torch.empty(B, plan.M, **f64),
           "weight": torch.empty(B, **f64), "info": torch.empty(B, dtype=torch.int32, device=dev)}
    x, a, f = td(xyz), td(aed), td(force)
    plan.solve_device(B, x, f, aed=a, out=fwd, shared_factor=shared_factor)
    res = {"joint_xyz": torch.empty(B, plan.nJ, plan.dim, **f64), "member_aed": torch.empty(B, plan.M, 3, **f64),
           "force": torch.empty(B, plan.N, **f64), "info": torch.empty(B, dtype=torch.int32, device=dev)}
    plan.adjoint_device(B, x, f, a, fwd["u"], {k: td(v) for k, v in grads.items()}, res, shared_factor=shared_factor)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in fwd.items()}, {k: v.cpu().numpy() for k, v in res.items()}


def random_grads(rng, B, N, M):
    return {"u": rng.standard_normal((B, N)), "ext": rng.standard_normal((B, N)), "axial": rng.standard_normal((B, M)),
            "weight": rng.standard_normal(B)}


def oracle_grads(dim, joints, support, conn, aed, force, grads, b):
    return adj.adjoint(dim, joints, support, conn, aed, force, g_u=grads["u"][b], g_ext=grads["ext"][b],
                       g_axial=grads["axial"][b], g_w=float(grads["weight"][b]))


def assert_grads_close(got, want, b, tol=1e-9, what=""):
    for k in FIELDS:
        err = orc.normwise_err(got[k][b], want[k])
        assert err <= tol, f"{what} system {b} field {k}: norm-wise err {err:.3e} > {tol:g}"
    for col, name in enumerate(("a", "e", "density")):      # the e column is ~1e-7 of the a column: checked on its own
        err = orc.normwise_err(got["member_aed"][b][:, col], want["member_aed"][:, col])
        assert err <= 100 * tol, f"{what} system {b} d/d{name}: norm-wise err {err:.3e}"


@PATHS
@pytest.mark.parametrize("name,dim,data,gold", H.shipped_cases(), ids=lambda v: v if isinstance(v, str) else None)
def test_adjoint_vs_oracle_every_fixture_every_path(name, dim, data, gold, path):
    joints, support, conn, aed, force = orc.arrays_from_json(data, dim)
    plan = _lib.Plan(dim, conn, support)
    force_path(plan, path)
    rng = np.random.default_rng(len(name) + 10 * path)
    B = 2
    aedb = np.repeat(aed[None], B, axis=0)
    aedb[1, :, 0] *= rng.uniform(0.5, 2.0, size=plan.M)           # a second sizing
    grads = random_grads(rng, B, plan.N, plan.M)
    fwd, got = device_adjoint(plan, joints, aedb, force, grads)
    assert not fwd["info"].any() and not got["info"].any()
    for b in range(B):
        assert_grads_close(got, oracle_grads(dim, joints, support, conn, aedb[b], force, grads, b), b, what=f"{name} path{path}")


def test_shared_factor_load_cases_bar942():
    t = Truss(3).LoadFromJSON(f"{H.GOLDEN}/ref_data/bar-942_input_0.json")
    joints, support, conn, aed, force = t._pack()
    plan = t._get_plan()
    assert plan.path == 2
    rng = np.random.default_rng(3)
    B = 64
    F = rng.uniform(-10.0, 10.0, size=(B, plan.N))
    grads = random_grads(rng, B, plan.N, plan.M)
    _, shared = device_adjoint(plan, joints, aed, F, grads, shared_factor=True)
    _, indep = device_adjoint(plan, joints, aed, F, grads)
    assert not shared["info"].any()
    for k in FIELDS:
        for b in range(B):
            assert orc.normwise_err(shared[k][b], indep[k][b]) <= 1e-10, (k, b)
    for b in (0, 37):
        assert_grads_close(shared, oracle_grads(3, joints, support, conn, aed, F[b], grads, b), b, what="bar-942 load cases")


@pytest.mark.parametrize("name", ["bar-72", "bar-942"])
def test_adjoint_is_deterministic_and_batch_independent(name):
    t = Truss(3).LoadFromJSON(f"{H.GOLDEN}/ref_data/{name}_input_0.json")
    joints, support, conn, aed, force = t._pack()
    plan = t._get_plan()
    rng = np.random.default_rng(11)
    B = 5
    xyzb = np.repeat(joints[None], B, axis=0) + rng.normal(0.0, 0.01, size=(B,) + joints.shape)
    aedb = np.repeat(aed[None], B, axis=0)
    aedb[:, :, 0] *= rng.uniform(0.5, 2.0, size=(B, plan.M))
    grads = random_grads(rng, B, plan.N, plan.M)
    _, one = device_adjoint(plan, xyzb, aedb, force, grads)
    _, two = device_adjoint(plan, xyzb, aedb, force, grads)
    for k in FIELDS:
        assert np.array_equal(one[k], two[k]), k
    for b in range(B):
        _, single = device_adjoint(plan, xyzb[b:b + 1], aedb[b:b + 1], force, {k: v[b:b + 1] for k, v in grads.items()})
        for k in FIELDS:
            assert np.array_equal(single[k][0], one[k][b]), (k, b)


def test_failed_systems_get_zero_gradients():
    data = json.load(open(f"{H.GOLDEN}/ref_data/bar-10_input_0.json"))
    joints, support, conn, aed, force = orc.arrays_from_json(data, 2)
    plan = _lib.Plan(2, conn, support)
    B = 6
    xyzb = np.repeat(joints[None], B, axis=0)
    aedb = np.repeat(aed[None], B, axis=0)
    j0, j1 = conn[0]
    xyzb[1, j1] = xyzb[1, j0]                                  # zero-length member
    aedb[3, :, 1] = 0.0                                        # no stiffness at all: singular K
    xyzb[5, :, 1] = 0.0                                        # every joint on one line: a mechanism (singular K)
    xyzb[5, :, 0] = np.arange(plan.nJ) * 100.0
    grads = random_grads(np.random.default_rng(5), B, plan.N, plan.M)
    _, got = device_adjoint(plan, xyzb, aedb, force, grads)
    good = [0, 2, 4]
    assert got["info"][1] == -2 and got["info"][3] > 0 and got["info"][5] > 0 and not got["info"][good].any()
    for k in FIELDS:
        assert np.isfinite(got[k]).all(), k
        assert not got[k][[1, 3, 5]].any(), k
    # the neighbours are the gradients of the same systems in a batch without failures
    _, clean = device_adjoint(plan, xyzb[good], aedb[good], force, {k: v[good] for k, v in grads.items()})
    for k in FIELDS:
        assert np.array_equal(clean[k], got[k][good]), k
    # a topology that fails the counting rule: every system fails
    bad = _lib.Plan(3, np.array([[0, 1]], np.int32), np.array([1, 0], np.uint8))
    _, g = device_adjoint(bad, np.array([[0.0, 0, 0], [1, 0, 0]]), np.array([[1.0, 1e7, 1.0]]), np.zeros(6),
                          random_grads(np.random.default_rng(0), 1, 6, 1))
    assert g["info"][0] == -1 and not any(g[k].any() for k in FIELDS)


@pytest.mark.parametrize("name", ["bar-6", "bar-10"])
def test_autograd_gradcheck(name):
    torch = _torch()
    from python_stable_3d_truss_analysis_b200 import autograd

    dim = H.dim_of(name + "_")
    t = Truss(dim).LoadFromJSON(f"{H.GOLDEN}/ref_data/{name}_input_0.json")
    joints, _, _, aed, force = t._pack()
    dev = torch.device("cuda:0")
    x0, a0, f0 = (torch.tensor(v, dtype=torch.float64, device=dev) for v in (joints, aed, force))
    ref = autograd.solve(t, x0, a0, f0)
    scale = {k: ref[k].abs().max() for k in ("u", "ext", "axial", "weight")}
    span = float(np.ptp(joints, axis=0).max())

    def fn(dx, sa, sf):                          # relative perturbations of every input; outputs O(1)
        out = autograd.solve(t, xyz=x0 + span * dx, aed=a0 * sa, force=f0 * sf)
        return tuple(out[k] / scale[k] for k in ("u", "ext", "axial", "weight"))

    args = (torch.zeros_like(x0, requires_grad=True), torch.ones_like(a0, requires_grad=True),
            torch.ones_like(f0, requires_grad=True))
    assert torch.autograd.gradcheck(fn, args, eps=1e-6, atol=1e-5, rtol=1e-3)
    # d(f.u)/df = u + K^-1 f = 2u (u and the loads' gradient vanish at supported DOFs)
    f = f0.clone().requires_grad_(True)
    out = autograd.solve(t, force=f)
    (f * out["u"]).sum().backward()
    assert orc.normwise_err(f.grad.cpu().numpy(), 2.0 * out["u"].detach().cpu().numpy()) <= 1e-12


def test_compliance_identity_bar72_x8192():
    """The GA-sized batch on the fused path: dC/dA_m = -N_m^2 L_m / (E_m A_m^2) for C = f.u, per system."""
    torch = _torch()
    from python_stable_3d_truss_analysis_b200 import autograd

    t = Truss(3).LoadFromJSON(f"{H.GOLDEN}/ref_data/bar-72_input_0.json")
    joints, _, conn, aed, force = t._pack()
    assert t._get_plan().path == 0
    B = 8192
    rng = np.random.default_rng(9)
    aedb = np.repeat(aed[None], B, axis=0)
    aedb[:, :, 0] = rng.uniform(0.1, 5.0, size=(B, aed.shape[0]))
    dev = torch.device("cuda:0")
    a = torch.tensor(aedb, device=dev, requires_grad=True)
    f = torch.tensor(force, device=dev)
    out = autograd.solve(t, aed=a, force=f)
    (f * out["u"]).sum().backward()
    assert not out["info"].any()
    L = np.sqrt(((joints[conn[:, 1]] - joints[conn[:, 0]]) ** 2).sum(axis=1))
    N = out["axial"].detach().cpu().numpy()
    want = -N ** 2 * L / (aedb[:, :, 1] * aedb[:, :, 0] ** 2)
    got = a.grad[:, :, 0].cpu().numpy()
    err = np.abs(got - want).max(axis=1) / np.abs(want).max(axis=1)
    assert err.max() <= 1e-9, err.max()


def test_cube12_tiled_path_hbm_member_vectors():
    """12^3 cube truss (M = 14868: the per-member vectors do not fit shared memory) on the tiled path, two systems."""
    t = H.cube_truss(12)
    joints, support, conn, aed, force = t._pack()
    plan = t._get_plan()
    assert plan.path == 1 and plan.M == 14868
    rng = np.random.default_rng(12)
    B = 2
    aedb = np.repeat(aed[None], B, axis=0)
    aedb[:, :, 0] = rng.uniform(1.0, 20.0, size=(B, plan.M))
    grads = random_grads(rng, B, plan.N, plan.M)
    _, got = device_adjoint(plan, joints, aedb, force, grads)
    assert not got["info"].any()
    for b in range(B):
        assert_grads_close(got, oracle_grads(3, joints, support, conn, aedb[b], force, grads, b), b, what="cube12")
