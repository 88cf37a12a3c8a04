"""Reverse mode of the modal analysis without a GPU: the numpy eigenvalue gradients (oracle/modal_adjoint.py eigval_grad) against
five-point central differences of the oracle's eigenvalues, a closed form, the identities that follow from the
homogeneity and invariances of K and M, the semantics of repeated eigenvalues, and the argument checks of
tb_modes_adjoint and autograd.modes."""
import ctypes as C
import functools

import numpy as np
import pytest

from oracle import modal
from oracle import modal_adjoint
from oracle import truss_oracle as orc
from python_stable_3d_truss_analysis_b200 import _lib
from tests import helpers as H

TOL_FD = 1e-6
TOL_ID = 1e-12
# fixture -> relative finite-difference step: bar-72's two lowest eigenvalues are 0.25 % apart even with joint masses, so
# its eigenvalues curve fast and want a small step; elsewhere a larger step keeps the rounding of lambda out of the small
# joint-mass gradients.
FD_CASES = {"bar-10_input_0": 1e-4, "bar-25_input_0": 1e-4, "bar-47_input_0": 1e-4, "bar-72_input_0": 1e-5,
            "cube-7_case_1": 1e-4}


def _has_cuda():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def fixtures():
    return [(n, d, data) for n, d, data, _ in H.shipped_cases() if not n.startswith("bar-942")] + \
        [(n, d, data) for n, d, data, _ in H.cube7_shipped()[:2]]


def arrays(name):
    for n, d, data in fixtures():
        if n == name:
            return (d,) + tuple(orc.arrays_from_json(data, d)[:4])
    raise KeyError(name)


def joint_masses(dim, joints, conn, aed):
    """The joint masses of tests/test_gpu_modes.py: they break the symmetries, so the lowest modes are simple."""
    return np.linspace(0.0, 3.0, len(joints)) * float(np.mean(modal.member_masses(dim, joints, conn, aed)))


def fd_gradient(dim, joints, support, conn, aed, jm, g, consistent, rel):
    """d(g . lambda[:k])/d(xyz, aed, joint mass) by five-point central differences of modal.modes.  The step is rel times
    the quantity's own signed value (rel times the truss's span, or the mean joint mass, where that value is 0)."""
    k = len(g)
    x0 = np.concatenate([joints.ravel(), aed.ravel(), jm])
    nx, na = joints.size, aed.size
    zero_step = np.empty_like(x0)
    zero_step[:nx] = np.ptp(joints, axis=0).max()
    zero_step[nx:nx + na] = 1.0
    zero_step[nx + na:] = max(float(np.mean(jm)), float(np.mean(modal.member_masses(dim, joints, conn, aed))))

    def f(x):
        r = modal.modes(dim, x[:nx].reshape(joints.shape), support, conn, x[nx:nx + na].reshape(aed.shape),
                        consistent=consistent, joint_mass=x[nx + na:])
        return g @ r["eigval_all"][:k]

    out = np.empty_like(x0)
    for i in range(x0.size):
        h = rel * (x0[i] if x0[i] != 0.0 else zero_step[i])
        e = np.zeros_like(x0)
        e[i] = h
        out[i] = (8.0 * (f(x0 + e) - f(x0 - e)) - (f(x0 + 2 * e) - f(x0 - 2 * e))) / (12.0 * h)
    return out[:nx].reshape(joints.shape), out[nx:nx + na].reshape(aed.shape), out[nx + na:]


def assert_fields_close(got, want, tol, what=""):
    for name, a, b in zip(("xyz", "aed", "joint_mass"), got, want):
        err = orc.normwise_err(np.ravel(a), np.ravel(b))
        assert err <= tol, f"{what} {name}: norm-wise err {err:.3e} > {tol:g}"


@pytest.mark.parametrize("consistent", [False, True], ids=["lumped", "consistent"])
@pytest.mark.parametrize("name", FD_CASES)
def test_eigval_grad_matches_finite_differences(name, consistent):
    dim, joints, support, conn, aed = arrays(name)
    jm = joint_masses(dim, joints, conn, aed)
    r = modal.modes(dim, joints, support, conn, aed, consistent=consistent, joint_mass=jm)
    k = min(6, len(r["eigval_all"]))
    assert all(len(c) == 1 for c in modal.clusters(r["eigval_all"][:k + 1], 1e-6)), "the lowest modes are simple"
    g = np.random.default_rng(list(FD_CASES).index(name)).standard_normal(k)
    got = modal_adjoint.eigval_grad(dim, joints, support, conn, aed, r["eigval"][:k], r["modes"][:k], g, consistent)
    want = fd_gradient(dim, joints, support, conn, aed, jm, g, consistent, FD_CASES[name])
    assert_fields_close(got, want, TOL_FD, name)


def test_single_bar_closed_forms():
    """The bar of test_modes_cpu.py (one free DOF, x of joint 1): lambda = 2E/(rho L^2) lumped, 3E/(rho L^2) consistent,
    (E a / L) / (rho a L / 2 + m0) with a point mass m0 on joint 1, differentiated by hand."""
    E, rho, a, L, m0 = 2.0e7, 0.3, 1.5, 7.0, 4.0
    joints = np.array([[0.0, 0.0], [L, 0.0]])
    support = np.array([orc.PIN, orc.ROLLER_Y], np.uint8)
    conn = np.array([[0, 1]], np.int32)
    aed = np.array([[a, E, rho]])
    for consistent, cst in ((False, 2.0), (True, 3.0)):
        r = modal.modes(2, joints, support, conn, aed, consistent=consistent)
        gx, ga, gm = modal_adjoint.eigval_grad(2, joints, support, conn, aed, r["eigval"], r["modes"], [1.0], consistent)
        lam = cst * E / (rho * L * L)
        assert ga[0] == pytest.approx([0.0, cst / (rho * L * L), -lam / rho], rel=1e-13, abs=1e-13 * lam)
        dx = 2.0 * lam / L                             # lambda ~ L^-2
        assert gx == pytest.approx(np.array([[dx, 0.0], [-dx, 0.0]]), rel=1e-13, abs=1e-13 * dx)
        phi2 = r["modes"][0, 2] ** 2
        assert gm == pytest.approx([0.0, -lam * phi2], rel=1e-13)
    r = modal.modes(2, joints, support, conn, aed, joint_mass=[0.0, m0])
    gx, ga, gm = modal_adjoint.eigval_grad(2, joints, support, conn, aed, r["eigval"], r["modes"], [1.0])
    k, m = E * a / L, rho * a * L / 2 + m0
    lam = k / m
    assert lam == pytest.approx(r["eigval"][0], rel=1e-13)
    want_a = [(E / L) / m - k * (rho * L / 2) / m ** 2, (a / L) / m, -k * (a * L / 2) / m ** 2]
    assert ga[0] == pytest.approx(want_a, rel=1e-12)
    dL = -k / L / m - k * (rho * a / 2) / m ** 2         # d lambda / d L
    assert gx == pytest.approx(np.array([[-dL, 0.0], [dL, 0.0]]), rel=1e-12, abs=1e-13 * abs(dL))
    assert gm == pytest.approx([0.0, -lam / m], rel=1e-12)


def identities(dim, joints, support, conn, aed, jm, L, grads):
    """The residuals of the exact identities of section 11 (DESIGN.md), each divided by |L|:
      sum a dL/da + sum mu dL/dmu = 0          (K and M both scale with a; mu scaled alike)
      sum E dL/dE = L                          (K scales with E)
      sum rho dL/drho + sum mu dL/dmu = -L     (M scales with rho and mu)
      sum x.dL/dx + sum mu dL/dmu = -2L        (K ~ 1/s, M ~ s under x -> s x, mu -> s mu)
      sum_J dL/dx_J = 0                        (translation)
      sum_J x_J x dL/dx_J = 0                  (3D rotation, when every support is a pin: a rotation moves the structure
                                               against a roller)"""
    gx, ga, gm = grads
    mu = np.zeros(len(joints)) if jm is None else jm
    r = [np.dot(aed[:, 0], ga[:, 0]) + np.dot(mu, gm), np.dot(aed[:, 1], ga[:, 1]) - L,
         np.dot(aed[:, 2], ga[:, 2]) + np.dot(mu, gm) + L, np.sum(joints * gx) + np.dot(mu, gm) + 2.0 * L,
         np.abs(gx.sum(axis=0)).max()]
    if dim == 3 and set(np.unique(support)) <= {orc.NO, orc.PIN}:
        r.append(np.abs(np.cross(joints, gx).sum(axis=0)).max())
    return np.abs(np.array(r)) / abs(L)


@pytest.mark.parametrize("consistent", [False, True], ids=["lumped", "consistent"])
@pytest.mark.parametrize("name", [f[0] for f in fixtures()])
def test_identities(name, consistent):
    dim, joints, support, conn, aed = arrays(name)
    for jm in (None, joint_masses(dim, joints, conn, aed)):
        r = modal.modes(dim, joints, support, conn, aed, consistent=consistent, joint_mass=jm)
        g = np.random.default_rng(5).uniform(0.5, 1.5, len(r["eigval"]))   # (positive: no cancellation in L)
        L = g @ r["eigval"]
        grads = modal_adjoint.eigval_grad(dim, joints, support, conn, aed, r["eigval"], r["modes"], g, consistent)
        assert identities(dim, joints, support, conn, aed, jm, L, grads).max() <= TOL_ID


def lowest_pair(lam):
    pair = [c for c in modal.clusters(lam, 1e-9) if len(c) > 1][0]
    assert len(pair) == 2 and pair[0] == 0, "the fixture's lowest eigenvalue is an exact pair"
    return pair


@functools.lru_cache(maxsize=None)
def _pair_case(name):
    dim, joints, support, conn, aed = arrays(name)
    r = modal.modes(dim, joints, support, conn, aed)
    return dim, joints, support, conn, aed, r, lowest_pair(r["eigval_all"])


@pytest.mark.parametrize("name", ["bar-72_input_0", "bar-120_input_0"])
def test_repeated_pair_sum_matches_finite_differences(name):
    dim, joints, support, conn, aed, r, pair = _pair_case(name)
    k = pair[-1] + 1
    g = np.ones(k)
    got = modal_adjoint.eigval_grad(dim, joints, support, conn, aed, r["eigval"][:k], r["modes"][:k], g)
    want = fd_gradient(dim, joints, support, conn, aed, np.zeros(len(joints)), g, False, 1e-5)
    assert_fields_close(got, want, TOL_FD, name)


def _rotated(modes_k, pair, theta=0.7):
    out = modes_k.copy()
    c, s = np.cos(theta), np.sin(theta)
    i, j = pair
    out[i], out[j] = c * modes_k[i] + s * modes_k[j], -s * modes_k[i] + c * modes_k[j]
    return out


@pytest.mark.parametrize("name", ["bar-72_input_0", "bar-120_input_0"])
def test_repeated_pair_semantics(name):
    """A cotangent equal across the pair gives a gradient that does not depend on the pair's basis; a cotangent on one
    eigenvalue of the pair does depend on it (which is why autograd.modes documents the cluster rule)."""
    dim, joints, support, conn, aed, r, pair = _pair_case(name)
    k = pair[-1] + 1
    lam, phi = r["eigval"][:k], r["modes"][:k]
    rot = _rotated(phi, pair)
    Mff, mask = r["M_ff"], r["mask"]
    assert np.abs(rot[:, mask] @ Mff @ rot[:, mask].T - np.eye(k)).max() <= 1e-12   # still an M-orthonormal basis
    both = np.zeros(k)
    both[pair] = 1.0
    a = modal_adjoint.eigval_grad(dim, joints, support, conn, aed, lam, phi, both)
    b = modal_adjoint.eigval_grad(dim, joints, support, conn, aed, lam, rot, both)
    assert_fields_close(b, a, 1e-12, "pair sum")
    one = np.zeros(k)
    one[pair[0]] = 1.0
    a1 = modal_adjoint.eigval_grad(dim, joints, support, conn, aed, lam, phi, one)
    b1 = modal_adjoint.eigval_grad(dim, joints, support, conn, aed, lam, rot, one)
    assert orc.normwise_err(b1[1].ravel(), a1[1].ravel()) > 1e-2, "a single eigenvalue of the pair is basis-dependent"


# ---- C ABI ---------------------------------------------------------------------------------------------------------
def _plan_and_inputs(name="bar-72_input_0"):
    data = H.load_json(f"ref_data/{name}.json")
    dim = H.dim_of(name)
    joints, support, conn, aed, _ = orc.arrays_from_json(data, dim)
    return _lib.Plan(dim, conn, support), joints, aed


def _buffers(plan, B, k):
    bufs = {"eigval": np.zeros((B, k)), "modes": np.zeros((B, k, plan.N)), "info": np.zeros(B, np.int32),
            "g": np.ones((B, k)), "gx": np.zeros((B, plan.nJ, plan.dim)), "ga": np.zeros((B, plan.M, 3)),
            "gm": np.zeros((B, plan.nJ))}
    ai = _lib.TbModesAdjIn(bufs["eigval"].ctypes.data, bufs["modes"].ctypes.data, bufs["info"].ctypes.data,
                           bufs["g"].ctypes.data)
    ao = _lib.TbModesAdjOut(bufs["gx"].ctypes.data, bufs["ga"].ctypes.data, bufs["gm"].ctypes.data)
    return bufs, ai, ao


def _call(plan_h, bi, mi, ai, ao):
    return _lib.lib().tb_modes_adjoint(plan_h, bi, mi, ai, ao, None)


def test_abi_structs_and_export():
    assert "tb_modes_adjoint" in _lib.EXPORTS
    assert [f[0] for f in _lib.TbModesAdjIn._fields_] == ["eigval", "modes", "info", "g_eigval"]
    assert [f[0] for f in _lib.TbModesAdjOut._fields_] == ["joint_xyz", "member_aed", "joint_mass"]


def test_argument_errors():
    plan, joints, aed = _plan_and_inputs()
    keep = []
    B, k = 2, 6
    bi = plan._batch_in(B, joints, aed, None, None, np.zeros(plan.N), keep)
    bi.force = None                                    # (not read)
    bufs, ai, ao = _buffers(plan, B, k)
    mi = _lib.TbModesIn(k, 0, None, 0)
    ref = C.byref
    assert _call(None, ref(bi), ref(mi), ref(ai), ref(ao)) == -1
    assert _call(plan._h, None, ref(mi), ref(ai), ref(ao)) == -1
    assert _call(plan._h, ref(bi), None, ref(ai), ref(ao)) == -1
    assert _call(plan._h, ref(bi), ref(mi), None, ref(ao)) == -1
    assert _call(plan._h, ref(bi), ref(mi), ref(ai), None) == -1
    for f in ("eigval", "modes", "info", "g_eigval"):  # every forward array and the cotangent are required
        bad = _lib.TbModesAdjIn.from_buffer_copy(ai)
        setattr(bad, f, None)
        assert _call(plan._h, ref(bi), ref(mi), ref(bad), ref(ao)) == -1, f
    for nm in (0, -1, plan.n + 1):
        assert _call(plan._h, ref(bi), ref(_lib.TbModesIn(nm, 0, None, 0)), ref(ai), ref(ao)) == -3
    assert _call(plan._h, ref(bi), ref(_lib.TbModesIn(k, 2, None, 0)), ref(ai), ref(ao)) == -3
    neg = _lib.TbBatchIn.from_buffer_copy(bi)
    neg.batch = -1
    assert _call(plan._h, ref(neg), ref(mi), ref(ai), ref(ao)) == -3
    table = np.array([[1.0, 1e7, 0.1]])                 # a gene / type-table batch has no member gradient
    gb = plan._batch_in(B, joints, None, np.zeros((B, plan.M), np.int32), table, np.zeros(plan.N), keep)
    assert _call(plan._h, ref(gb), ref(mi), ref(ai), ref(ao)) == -1
    nx = _lib.TbBatchIn.from_buffer_copy(bi)
    nx.joint_xyz = None
    assert _call(plan._h, ref(nx), ref(mi), ref(ai), ref(ao)) == -1
    empty = _lib.TbBatchIn.from_buffer_copy(bi)        # an empty batch is a no-op once the arguments are valid
    empty.batch = 0
    assert _call(plan._h, ref(empty), ref(mi), ref(ai), ref(ao)) in (0, _lib.TB_ERR_NO_DEVICE)
    skip = _lib.TbModesAdjOut(None, None, None)         # every output may be skipped
    assert _call(plan._h, ref(empty), ref(mi), ref(ai), ref(skip)) in (0, _lib.TB_ERR_NO_DEVICE)


def test_bar942_is_too_large():
    plan, joints, aed = _plan_and_inputs("bar-942_input_0")
    assert plan.n > 160
    keep = []
    bi = plan._batch_in(1, joints, aed, None, None, np.zeros(plan.N), keep)
    bufs, ai, ao = _buffers(plan, 1, 6)
    assert _call(plan._h, C.byref(bi), C.byref(_lib.TbModesIn(6, 0, None, 0)), C.byref(ai), C.byref(ao)) == \
        _lib.TB_ERR_TOO_LARGE


@pytest.mark.skipif(_has_cuda(), reason="only meaningful on a machine without a GPU")
def test_no_device():
    plan, joints, aed = _plan_and_inputs()
    keep = []
    bi = plan._batch_in(3, joints, aed, None, None, np.zeros(plan.N), keep)
    bufs, ai, ao = _buffers(plan, 3, 6)
    for consistent in (0, 1):
        assert _call(plan._h, C.byref(bi), C.byref(_lib.TbModesIn(6, consistent, None, 0)), C.byref(ai), C.byref(ao)) == \
            _lib.TB_ERR_NO_DEVICE


def test_autograd_argument_types():
    """dtype and device are checked before anything runs (shapes and batch sizes: tests/test_gpu_modes_adjoint.py,
    which has CUDA tensors to pass)."""
    torch = pytest.importorskip("torch")
    from python_stable_3d_truss_analysis_b200 import autograd
    from python_stable_3d_truss_analysis_b200.truss import Truss

    t = Truss(3).LoadFromJSON(data=H.load_json("ref_data/bar-72_input_0.json"))
    joints, _, _, aed, _ = t._pack()
    with pytest.raises(TypeError):
        autograd.modes(t, xyz=torch.tensor(joints, dtype=torch.float32))
    with pytest.raises(TypeError):
        autograd.modes(t, aed=torch.tensor(aed, dtype=torch.float64))            # a CPU tensor
    with pytest.raises(TypeError):
        autograd.modes(t, joint_mass=torch.ones(t.nJoint, dtype=torch.float64))   # a CPU tensor
