"""Reverse mode of the solve without a GPU: the numpy adjoint (oracle/adjoint.py) against central differences of the
oracle's forward solve, two identities it must satisfy, and the argument checks of tb_adjoint."""
import ctypes as C
import functools
import json

import numpy as np
import pytest

from oracle import adjoint as adj
from oracle import truss_oracle as orc
from python_stable_3d_truss_analysis_b200 import _lib
from tests import helpers as H

TOL = 1e-6


def random_truss(dim, seed):
    """A complete graph over a few random joints (rigid), supported by every support type of the dimension plus a second
    pin (statically indeterminate, so the reactions depend on the member stiffnesses), with loads on every joint, the
    supported ones included."""
    rng = np.random.default_rng(seed)
    nJ = 6 if dim == 2 else 7
    joints = rng.uniform(-100.0, 100.0, size=(nJ, dim))
    support = [orc.PIN, orc.ROLLER_X, orc.ROLLER_Y] + ([orc.ROLLER_Z] if dim == 3 else []) + [orc.PIN]
    support = np.array(support + [orc.NO] * (nJ - len(support)), np.uint8)
    conn = np.array([(i, j) for i in range(nJ) for j in range(i + 1, nJ)], np.int32)
    if seed % 2:
        conn = conn[:, ::-1].copy()              # members pointing both ways
    aed = np.stack([rng.uniform(1.0, 5.0, len(conn)), rng.uniform(1e7, 3e7, len(conn)), rng.uniform(0.1, 1.0, len(conn))], 1)
    force = rng.uniform(-1000.0, 1000.0, size=nJ * dim)
    return joints, support, conn, aed, force


def case(name):
    if name.startswith("random"):
        dim, seed = int(name[6]), int(name.split("_")[1])
        return (dim,) + random_truss(dim, seed)
    dim = H.dim_of(name + "_")
    data = json.load(open(f"{H.GOLDEN}/ref_data/{name}_input_0.json"))
    return (dim,) + orc.arrays_from_json(data, dim)


CASES = ["bar-6", "bar-10", "bar-25", "bar-72", "random2_1", "random2_2", "random3_3", "random3_4"]


@functools.lru_cache(maxsize=None)
def fd_jacobian(name):
    """d(u, ext, axial, weight)/d(xyz, aed, force) by five-point central differences of truss_oracle.solve; the step is
    1e-3 of each quantity's scale (span of the truss, largest a / e / density, largest load)."""
    dim, joints, support, conn, aed, force = case(name)
    nx, na = joints.size, aed.size
    x0 = np.concatenate([joints.ravel(), aed.ravel(), force])
    scale = np.empty_like(x0)
    scale[:nx] = np.ptp(joints, axis=0).max()
    for col in range(3):
        scale[nx + col:nx + na:3] = np.abs(aed[:, col]).max()
    scale[nx + na:] = max(np.abs(force).max(), 1.0)

    def outs(x):
        r = orc.solve(dim, x[:nx].reshape(joints.shape), support, conn, x[nx:nx + na].reshape(aed.shape), x[nx + na:])
        return np.concatenate([r["u"], r["ext"], r["axial"], [r["weight"]]])

    cols = []
    for i in range(x0.size):
        h = 1e-3 * scale[i]
        e = np.zeros_like(x0)
        e[i] = h
        cols.append((8.0 * (outs(x0 + e) - outs(x0 - e)) - (outs(x0 + 2 * e) - outs(x0 - 2 * e))) / (12.0 * h))
    return np.array(cols).T


def cotangents(dim, nJ, M, which, seed):
    rng = np.random.default_rng(seed)
    N = dim * nJ
    return {"g_u": rng.standard_normal(N) if which in ("u", "all") else None,
            "g_ext": rng.standard_normal(N) if which in ("ext", "all") else None,
            "g_axial": rng.standard_normal(M) if which in ("axial", "all") else None,
            "g_w": float(rng.standard_normal()) if which in ("weight", "all") else 0.0}


WHICH = ["u", "ext", "axial", "weight", "all"]


@pytest.mark.parametrize("which", WHICH)
@pytest.mark.parametrize("name", CASES)
def test_numpy_adjoint_matches_finite_differences(name, which):
    dim, joints, support, conn, aed, force = case(name)
    nJ, M, N = joints.shape[0], conn.shape[0], force.size
    g = cotangents(dim, nJ, M, which, seed=10 * CASES.index(name) + WHICH.index(which))
    vec = np.concatenate([g["g_u"] if g["g_u"] is not None else np.zeros(N), g["g_ext"] if g["g_ext"] is not None else np.zeros(N),
                          g["g_axial"] if g["g_axial"] is not None else np.zeros(M), [g["g_w"]]])
    fd = vec @ fd_jacobian(name)
    got = adj.adjoint(dim, joints, support, conn, aed, force, **g)
    nx, na = joints.size, aed.size
    assert orc.normwise_err(got["joint_xyz"].ravel(), fd[:nx]) <= TOL, "xyz"
    fd_aed = fd[nx:nx + na].reshape(-1, 3)
    for col, what in enumerate(("a", "e", "density")):
        if np.any(fd_aed[:, col]) or np.any(got["member_aed"][:, col]):
            assert orc.normwise_err(got["member_aed"][:, col], fd_aed[:, col]) <= TOL, what
    if np.any(fd[nx + na:]) or np.any(got["force"]):
        assert orc.normwise_err(got["force"], fd[nx + na:]) <= TOL, "force"
    assert not np.any(got["force"][~orc.free_mask(dim, support)])     # loads on supported DOFs are overwritten


@pytest.mark.parametrize("name", CASES)
def test_compliance_identity(name):
    """C = f.u with f fixed: dC/dA_m = -N_m^2 L_m / (E_m A_m^2), and dC/df through u alone is u."""
    dim, joints, support, conn, aed, force = case(name)
    mask = orc.free_mask(dim, support)
    f = np.where(mask, force, 0.0)
    got = adj.adjoint(dim, joints, support, conn, aed, force, g_u=f)
    ref = orc.solve_closed_form(dim, joints, support, conn, aed, force)
    L = np.sqrt(((joints[conn[:, 1]] - joints[conn[:, 0]]) ** 2).sum(axis=1))
    want = -ref["axial"] ** 2 * L / (aed[:, 1] * aed[:, 0] ** 2)
    assert orc.normwise_err(got["member_aed"][:, 0], want) <= 1e-9
    assert orc.normwise_err(got["lam"], ref["u"]) <= 1e-9            # the adjoint of the compliance is u itself
    assert orc.normwise_err(got["force"], ref["u"]) <= 1e-9


@pytest.mark.parametrize("name", CASES)
def test_geometry_gradient_is_translation_invariant(name):
    """Moving every joint by the same vector changes nothing: the joint gradients sum to zero."""
    dim, joints, support, conn, aed, force = case(name)
    g = cotangents(dim, joints.shape[0], conn.shape[0], "all", seed=7)
    got = adj.adjoint(dim, joints, support, conn, aed, force, **g)
    tot = got["joint_xyz"].sum(axis=0)
    assert np.abs(tot).max() <= 1e-9 * np.abs(got["joint_xyz"]).max()


def _has_cuda():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def _adjoint_call(plan_h, bi, u=None):
    L = _lib.lib()
    gi, go = _lib.TbAdjIn(), _lib.TbAdjOut()
    return L.tb_adjoint(plan_h, bi, u, C.byref(gi), C.byref(go), 0, None)


def test_adjoint_argument_errors():
    dim, joints, support, conn, aed, force = case("bar-6")
    plan = _lib.Plan(dim, conn, support)
    keep = []
    bi = plan._batch_in(1, joints, aed, None, None, force, keep)
    assert _adjoint_call(None, C.byref(bi)) == -1                     # null plan
    assert _adjoint_call(plan._h, None) == -1                         # null batch
    gene = plan._batch_in(1, joints, None, np.zeros(plan.M, np.int32), np.array([[1.0, 1e7, 0.1]]), force, keep)
    assert _adjoint_call(plan._h, C.byref(gene)) == -1                # a type-table batch has no member gradient


@pytest.mark.skipif(_has_cuda(), reason="only meaningful on a machine without a GPU")
def test_adjoint_without_a_device():
    dim, joints, support, conn, aed, force = case("bar-6")
    plan = _lib.Plan(dim, conn, support)
    keep = []
    bi = plan._batch_in(1, joints, aed, None, None, force, keep)
    u = np.zeros(plan.N)
    assert _adjoint_call(plan._h, C.byref(bi), u.ctypes.data) == _lib.TB_ERR_NO_DEVICE
