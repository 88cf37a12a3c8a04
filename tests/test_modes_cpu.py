"""Modal analysis without a GPU: the numpy restatement (oracle/modal.py) against closed forms and scipy on every fixture,
and the argument checks of tb_modes / tb_modes_host."""
import ctypes as C

import numpy as np
import pytest

from oracle import modal
from oracle import truss_oracle as orc
from python_stable_3d_truss_analysis_b200 import _lib
from tests import helpers as H


def _has_cuda():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def bar(E=2.0e7, rho=0.3, a=1.5, L=7.0):
    """2D bar from a pin to a ROLLER_Y joint: one free DOF (x of joint 1)."""
    joints = np.array([[0.0, 0.0], [L, 0.0]])
    support = np.array([orc.PIN, orc.ROLLER_Y], np.uint8)
    return joints, support, np.array([[0, 1]], np.int32), np.array([[a, E, rho]])


def chain(n, E=3.0e7, rho=0.2, a=2.0, L=5.0):
    """Fixed-fixed chain of n equal 2D bars along x; the interior joints move along x only (ROLLER_Y)."""
    joints = np.stack([np.arange(n + 1) * L, np.zeros(n + 1)], 1)
    support = np.array([orc.PIN] + [orc.ROLLER_Y] * (n - 1) + [orc.PIN], np.uint8)
    conn = np.array([(i, i + 1) for i in range(n)], np.int32)
    return joints, support, conn, np.tile([a, E, rho], (n, 1))


def fixtures():
    return [(n, d, data) for n, d, data, _ in H.shipped_cases() if not n.startswith("bar-942")] + \
        [(n, d, data) for n, d, data, _ in H.cube7_shipped()[:2]]


def test_single_bar_closed_forms():
    E, rho, a, L = 2.0e7, 0.3, 1.5, 7.0
    j, s, c, aed = bar(E, rho, a, L)
    lum = modal.modes(2, j, s, c, aed)
    con = modal.modes(2, j, s, c, aed, consistent=True)
    assert lum["eigval"][0] == pytest.approx(2 * E / (rho * L * L), rel=1e-13)
    assert con["eigval"][0] == pytest.approx(3 * E / (rho * L * L), rel=1e-13)
    m0 = 4.0                                           # a point mass on the free joint
    jm = modal.modes(2, j, s, c, aed, joint_mass=[0.0, m0])
    assert jm["eigval"][0] == pytest.approx((E * a / L) / (rho * a * L / 2 + m0), rel=1e-13)
    # one free DOF: the mode is +1/sqrt(m) on x of joint 1, zero elsewhere
    assert np.allclose(lum["modes"][0], [0, 0, 1 / np.sqrt(rho * a * L / 2), 0], rtol=1e-13)


@pytest.mark.parametrize("n", [2, 3, 8, 17])
def test_chain_closed_form(n):
    E, rho, a, L = 3.0e7, 0.2, 2.0, 5.0
    k, m = E * a / L, rho * a * L
    j, s, c, aed = chain(n, E, rho, a, L)
    jj = np.arange(1, n)
    want = 4 * k / m * np.sin(jj * np.pi / (2 * n)) ** 2
    got = modal.modes(2, j, s, c, aed)
    assert np.allclose(got["eigval"], want, rtol=1e-12, atol=0)
    m0 = 0.7 * m                                       # the same point mass on every joint
    got = modal.modes(2, j, s, c, aed, joint_mass=np.full(n + 1, m0))
    assert np.allclose(got["eigval"], 4 * k / (m + m0) * np.sin(jj * np.pi / (2 * n)) ** 2, rtol=1e-12, atol=0)
    # the mode shapes are sines: phi_j(i) ~ sin(i j pi / n) at interior joint i (up to sign: several components of a
    # sine can have the same magnitude, and then rounding decides which one the sign convention sees first)
    phi = got["modes"][:, 0::2][:, 1:n]
    for q in range(n - 1):
        ref = np.sin(np.arange(1, n) * (q + 1) * np.pi / n)
        ref = ref / np.abs(ref).max() * np.sign(ref @ phi[q])
        assert np.allclose(phi[q] / np.abs(phi[q]).max(), ref, atol=1e-10)


@pytest.mark.parametrize("consistent", [False, True], ids=["lumped", "consistent"])
@pytest.mark.parametrize("name,dim,data", fixtures(), ids=[f[0] for f in fixtures()])
def test_oracle_against_eigh(name, dim, data, consistent):
    joints, support, conn, aed, _ = orc.arrays_from_json(data, dim)
    jm = np.linspace(0.0, 3.0, len(joints)) * float(np.mean(modal.member_masses(dim, joints, conn, aed)))
    for joint_mass in (None, jm):
        r = modal.modes(dim, joints, support, conn, aed, consistent=consistent, joint_mass=joint_mass)
        K, Mf, mask = r["K_ff"], r["M_ff"], r["mask"]
        lam, phi = r["eigval"], r["modes"][:, mask].T
        lmax = np.abs(r["eigval_all"]).max()
        res = K @ phi - (Mf @ phi) * lam
        assert np.abs(res).max() <= 1e-12 * lmax * np.abs(Mf @ phi).max()
        assert np.abs(phi.T @ Mf @ phi - np.eye(len(lam))).max() <= 1e-12
        assert np.all(np.diff(lam) >= 0)
        assert np.all(r["modes"][:, ~mask] == 0.0)
        big = np.argmax(np.abs(phi), axis=0)
        assert np.all(phi[big, np.arange(phi.shape[1])] > 0)
        if not consistent:                             # total lumped mass before the supports are removed
            Mall = modal.mass_matrix(dim, joints, conn, aed, joint_mass=joint_mass)
            total = dim * (modal.member_masses(dim, joints, conn, aed).sum() + (0 if joint_mass is None else jm.sum()))
            assert np.trace(Mall) == pytest.approx(total, rel=1e-13)
            assert np.count_nonzero(Mall - np.diag(np.diag(Mall))) == 0
        else:
            assert np.abs(Mf - Mf.T).max() == 0.0


def test_oracle_K_is_the_static_solves():
    name, dim, data, _ = H.shipped_cases()[0]
    joints, support, conn, aed, _ = orc.arrays_from_json(data, dim)
    r = modal.modes(dim, joints, support, conn, aed)
    K = orc.assemble_K(dim, joints, conn, aed)
    assert np.array_equal(r["K_ff"], K[np.ix_(r["mask"], r["mask"])])


def test_info_codes_and_exports():
    assert (_lib.TB_INFO_MASS, _lib.TB_INFO_NO_CONVERGENCE) == (-5, -6)
    assert {"tb_modes", "tb_modes_host"} <= set(_lib.EXPORTS)
    assert [f[0] for f in _lib.TbModesIn._fields_] == ["n_modes", "consistent", "joint_mass", "joint_mass_stride"]
    assert [f[0] for f in _lib.TbModesOut._fields_] == ["eigval", "modes", "info"]


def _plan_and_inputs(name="bar-72_input_0"):
    data = H.load_json(f"ref_data/{name}.json")
    dim = H.dim_of(name)
    joints, support, conn, aed, _ = orc.arrays_from_json(data, dim)
    plan = _lib.Plan(dim, conn, support)
    return plan, joints, aed


def _call(plan, bi, mi, mo, host):
    L = _lib.lib()
    if host:
        return L.tb_modes_host(plan._h, bi, mi, mo)
    return L.tb_modes(plan._h, bi, mi, mo, None)


@pytest.mark.parametrize("host", [False, True], ids=["device", "host"])
def test_argument_errors(host):
    plan, joints, aed = _plan_and_inputs()
    keep = []
    B = 2
    bi = plan._batch_in(B, joints, aed, None, None, np.zeros(plan.N), keep)
    bi.force = None                                    # (ignored by tb_modes)
    ev, modes, info = np.zeros((B, plan.n)), np.zeros((B, plan.n, plan.N)), np.zeros(B, np.int32)
    mo = _lib.TbModesOut(ev.ctypes.data, modes.ctypes.data, info.ctypes.data)
    mi = _lib.TbModesIn(6, 0, None, 0)
    ref = C.byref
    assert _call(plan, ref(bi), None, ref(mo), host) == -1                     # m
    assert _call(plan, ref(bi), ref(mi), None, host) == -1
    assert _call(plan, ref(bi), ref(mi), ref(_lib.TbModesOut(None, modes.ctypes.data, info.ctypes.data)), host) == -1
    assert _call(plan, ref(bi), ref(mi), ref(_lib.TbModesOut(ev.ctypes.data, modes.ctypes.data, None)), host) == -1
    for nm in (0, -1, plan.n + 1):
        assert _call(plan, ref(bi), ref(_lib.TbModesIn(nm, 0, None, 0)), ref(mo), host) == -3
    assert _call(plan, ref(bi), ref(_lib.TbModesIn(6, 2, None, 0)), ref(mo), host) == -3
    bad = _lib.TbBatchIn.from_buffer_copy(bi)
    bad.batch = -1
    assert _call(plan, ref(bad), ref(mi), ref(mo), host) == -3
    gene = np.zeros((B, plan.M), np.int32)             # a gene batch without a type table
    gb = _lib.TbBatchIn.from_buffer_copy(bi)
    gb.member_aed, gb.gene, gb.gene_stride, gb.type_table, gb.n_type = None, gene.ctypes.data, plan.M, None, 0
    assert _call(plan, ref(gb), ref(mi), ref(mo), host) == -1
    nx = _lib.TbBatchIn.from_buffer_copy(bi)
    nx.joint_xyz = None
    assert _call(plan, ref(nx), ref(mi), ref(mo), host) == -1
    empty = _lib.TbBatchIn.from_buffer_copy(bi)        # an empty batch is a no-op once the arguments are valid
    empty.batch = 0
    rc = _call(plan, ref(empty), ref(mi), ref(mo), host)
    assert rc in (0, _lib.TB_ERR_NO_DEVICE)


@pytest.mark.parametrize("host", [False, True], ids=["device", "host"])
def test_bar942_is_too_large(host):
    plan, joints, aed = _plan_and_inputs("bar-942_input_0")
    assert plan.n > 160
    keep = []
    bi = plan._batch_in(1, joints, aed, None, None, np.zeros(plan.N), keep)
    ev, info = np.zeros((1, 6)), np.zeros(1, np.int32)
    mo = _lib.TbModesOut(ev.ctypes.data, None, info.ctypes.data)
    assert _call(plan, C.byref(bi), C.byref(_lib.TbModesIn(6, 0, None, 0)), C.byref(mo), host) == _lib.TB_ERR_TOO_LARGE
    with pytest.raises(_lib.TrussLibError) as e:
        plan.modes_host(1, joints, aed=aed, n_modes=6)
    assert e.value.code == _lib.TB_ERR_TOO_LARGE


@pytest.mark.skipif(_has_cuda(), reason="only meaningful on a machine without a GPU")
def test_no_device():
    plan, joints, aed = _plan_and_inputs()
    with pytest.raises(_lib.NoCudaDeviceError):
        plan.modes_host(3, joints, aed=aed, n_modes=6)
    with pytest.raises(_lib.NoCudaDeviceError):
        plan.modes_host(1, joints, aed=aed, consistent=True, joint_mass=np.ones(plan.nJ))
    from python_stable_3d_truss_analysis_b200.truss import Truss
    t = Truss(3).LoadFromJSON(data=H.load_json("ref_data/bar-72_input_0.json"))
    with pytest.raises(_lib.NoCudaDeviceError):
        t.SolveModes(6)
    with pytest.raises(Exception):
        t.GetEigenvalues()


def test_python_arguments():
    plan, joints, aed = _plan_and_inputs()
    with pytest.raises(ValueError):
        plan.modes_host(2, joints, aed=aed, joint_mass=np.ones(plan.nJ + 1))
    from python_stable_3d_truss_analysis_b200.batch import ModesBatch
    from python_stable_3d_truss_analysis_b200.truss import Truss
    t = Truss(3).LoadFromJSON(data=H.load_json("ref_data/bar-72_input_0.json"))
    with pytest.raises(ValueError):
        ModesBatch(t)                                  # neither aed nor genes
