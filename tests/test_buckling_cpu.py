"""Linear buckling without a GPU: the numpy restatement (oracle/buckling.py) against closed forms and against the direct
form on every fixture, and the argument checks of tb_buckling / tb_buckling_host."""
import ctypes as C

import numpy as np
import pytest

from oracle import buckling as bk
from oracle import truss_oracle as orc
from python_stable_3d_truss_analysis_b200 import _lib
from tests import helpers as H


def _has_cuda():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def braced_column(dim, E=2.0e7, A=1.5, Es=3.0e7, As=0.25, L=4.0, b=3.0, P=1.0e3):
    """A pinned column J0-J1 of height L, its top J1 held sideways by pinned braces of length b (one along x in 2D, one
    along x and one along y in 3D), loaded by P downwards at J1.  (joints, support, conn, aed, force)"""
    if dim == 2:
        joints = np.array([[0.0, 0.0], [0.0, L], [b, L]])
        support = np.array([orc.PIN, orc.NO, orc.PIN], np.uint8)
        conn = np.array([[0, 1], [2, 1]], np.int32)
        aed = np.array([[A, E, 0.1], [As, Es, 0.1]])
    else:
        joints = np.array([[0.0, 0.0, 0.0], [0.0, 0.0, L], [b, 0.0, L], [0.0, b, L]])
        support = np.array([orc.PIN, orc.NO, orc.PIN, orc.PIN], np.uint8)
        conn = np.array([[0, 1], [2, 1], [3, 1]], np.int32)
        aed = np.array([[A, E, 0.1], [As, Es, 0.1], [As, Es, 0.1]])
    force = np.zeros(len(joints) * dim)
    force[dim + dim - 1] = -P
    return joints, support, conn, aed, force


def axial_of(dim, joints, support, conn, aed, force):
    return orc.solve(dim, joints, support, conn, aed, force)["axial"]


def fixtures():
    """Every shipped fixture up to 160 free DOFs and two cube-7 cases, with its own loads."""
    return [(n, d, data) for n, d, data, _ in H.shipped_cases() if not n.startswith("bar-942")] + \
        [(n, d, data) for n, d, data, _ in H.cube7_shipped()[:2]]


@pytest.mark.parametrize("dim", [2, 3])
def test_braced_column_closed_form(dim):
    Es, As, L, b, P = 3.0e7, 0.25, 4.0, 3.0, 1.0e3
    j, s, c, aed, f = braced_column(dim, Es=Es, As=As, L=L, b=b, P=P)
    ax = axial_of(dim, j, s, c, aed, f)
    assert ax[0] == pytest.approx(-P, rel=1e-13) and np.all(ax[1:] == 0.0)
    r = bk.buckling(dim, j, s, c, aed, ax)
    lam = Es * As * L / (b * P)
    nfin = dim - 1                                     # one critical mode per braced direction
    assert np.allclose(r["factor"][:nfin], lam, rtol=1e-12, atol=0)
    assert np.all(np.isinf(r["factor"][nfin:]))
    assert np.all(r["modes"][nfin:] == 0.0)
    if dim == 2:                                       # phi_1 = (1 / sqrt(Es As / b), 0) at J1
        assert np.allclose(r["modes"][0], [0, 0, 1 / np.sqrt(Es * As / b), 0, 0, 0], rtol=1e-13, atol=0)
    else:                                              # a repeated pair spanning x and y of J1
        phi = r["modes"][:2][:, 3:5]
        assert np.allclose(phi @ phi.T, np.eye(2) / (Es * As / b), rtol=1e-12, atol=1e-20)
        assert np.all(r["modes"][:2][:, [0, 1, 2, 5]] == 0.0) and np.all(r["modes"][:2][:, 6:] == 0.0)


@pytest.mark.parametrize("dim", [2, 3])
def test_reversed_and_scaled_loads(dim):
    j, s, c, aed, f = braced_column(dim)
    ax = axial_of(dim, j, s, c, aed, f)
    assert np.all(np.isinf(bk.buckling(dim, j, s, c, aed, -ax)["factor"]))     # a pulled column never buckles
    assert np.all(np.isinf(bk.buckling(dim, j, s, c, aed, 0.0 * ax)["factor"]))
    base = bk.buckling(dim, j, s, c, aed, ax)["factor"]
    for sc in (0.5, 3.0, 1e4):
        got = bk.buckling(dim, j, s, c, aed, sc * ax)["factor"]
        fin = np.isfinite(base)
        assert np.array_equal(np.isfinite(got), fin)
        assert np.allclose(got[fin], base[fin] / sc, rtol=1e-12, atol=0)


def test_geometric_stiffness_form():
    """Symmetric, zero row sums (a rigid translation carries no geometric stiffness), c is in its null space per member,
    and linear in N."""
    name, dim, data = fixtures()[0]
    joints, support, conn, aed, force = orc.arrays_from_json(data, dim)
    ax = axial_of(dim, joints, support, conn, aed, force)
    KG = bk.geometric_stiffness(dim, joints, conn, ax)
    assert np.array_equal(KG, KG.T)
    assert np.abs(KG.reshape(KG.shape[0], -1, dim).sum(axis=1)).max() <= 1e-12 * np.abs(KG).max()
    one = bk.geometric_stiffness(dim, joints, conn[:1], ax[:1])
    j0, j1 = conn[0]
    d = joints[j1] - joints[j0]
    v = np.zeros(KG.shape[0])
    v[j1 * dim:(j1 + 1) * dim] = d                     # stretching member 0 along its axis: no geometric stiffness
    assert np.abs(one @ v).max() <= 1e-12 * np.abs(one).max() * np.linalg.norm(d)
    assert np.abs(bk.geometric_stiffness(dim, joints, conn, 2.5 * ax) - 2.5 * KG).max() <= 1e-14 * np.abs(2.5 * KG).max()


def _all_cases():
    out = [(f"braced-column-{d}d", d) + braced_column(d) for d in (2, 3)]
    for name, dim, data in fixtures():
        out.append((name, dim) + tuple(orc.arrays_from_json(data, dim)))
    return out


@pytest.mark.parametrize("case", _all_cases(), ids=[c[0] for c in _all_cases()])
def test_oracle_against_the_direct_form(case):
    name, dim, joints, support, conn, aed, force = case
    ax = axial_of(dim, joints, support, conn, aed, force)
    r = bk.buckling(dim, joints, support, conn, aed, ax)
    K, KG, mask = r["K_ff"], r["K_G_ff"], r["mask"]
    nu, lam = r["nu"], r["factor"]
    assert np.all(np.diff(nu) >= 0)
    fin = np.isfinite(lam)
    assert np.array_equal(fin, r["critical"])
    assert np.all(np.diff(lam[fin]) >= 0) and np.all(lam[fin] > 0)
    assert np.all(r["modes"][:, ~mask] == 0.0) and np.all(r["modes"][~fin] == 0.0)
    phi = r["modes"][fin][:, mask].T
    if phi.size:
        assert np.abs(phi.T @ K @ phi - np.eye(phi.shape[1])).max() <= 1e-12
        big = np.argmax(np.abs(phi), axis=0)
        assert np.all(phi[big, np.arange(phi.shape[1])] > 0)
    # K_ff + lambda_q K_G,ff is singular: its smallest singular value against the largest of K_ff
    smax = np.linalg.norm(K, 2)
    for q in np.nonzero(fin)[0][:6]:
        smin = np.linalg.svd(K + lam[q] * KG, compute_uv=False)[-1]
        assert smin <= 1e-10 * smax, (name, q, smin / smax)


def test_exports_and_structures():
    assert {"tb_buckling", "tb_buckling_host"} <= set(_lib.EXPORTS)
    assert [f[0] for f in _lib.TbBucklingIn._fields_] == ["n_modes", "axial", "axial_stride"]
    assert [f[0] for f in _lib.TbBucklingOut._fields_] == ["factor", "modes", "info"]


def _plan_and_inputs(name="bar-72_input_0"):
    data = H.load_json(f"ref_data/{name}.json")
    dim = H.dim_of(name)
    joints, support, conn, aed, _ = orc.arrays_from_json(data, dim)
    plan = _lib.Plan(dim, conn, support)
    return plan, joints, aed


def _call(plan, bi, bki, bo, host):
    L = _lib.lib()
    if host:
        return L.tb_buckling_host(plan._h, bi, bki, bo)
    return L.tb_buckling(plan._h, bi, bki, bo, None)


@pytest.mark.parametrize("host", [False, True], ids=["device", "host"])
def test_argument_errors(host):
    plan, joints, aed = _plan_and_inputs()
    keep = []
    B = 2
    bi = plan._batch_in(B, joints, aed, None, None, np.zeros(plan.N), keep)
    bi.force = None                                    # (ignored by tb_buckling)
    ax = np.zeros((B, plan.M))
    fac, modes, info = np.zeros((B, plan.n)), np.zeros((B, plan.n, plan.N)), np.zeros(B, np.int32)
    bo = _lib.TbBucklingOut(fac.ctypes.data, modes.ctypes.data, info.ctypes.data)
    bki = _lib.TbBucklingIn(6, ax.ctypes.data, plan.M)
    ref = C.byref
    assert _call(plan, ref(bi), None, ref(bo), host) == -1                     # bk
    assert _call(plan, ref(bi), ref(bki), None, host) == -1
    assert _call(plan, None, ref(bki), ref(bo), host) == -1
    assert _call(plan, ref(bi), ref(_lib.TbBucklingIn(6, None, plan.M)), ref(bo), host) == -1                # axial
    assert _call(plan, ref(bi), ref(bki), ref(_lib.TbBucklingOut(None, modes.ctypes.data, info.ctypes.data)), host) == -1
    assert _call(plan, ref(bi), ref(bki), ref(_lib.TbBucklingOut(fac.ctypes.data, modes.ctypes.data, None)), host) == -1
    for nm in (0, -1, plan.n + 1):
        assert _call(plan, ref(bi), ref(_lib.TbBucklingIn(nm, ax.ctypes.data, plan.M)), ref(bo), host) == -3
    assert _call(plan, ref(bi), ref(_lib.TbBucklingIn(6, ax.ctypes.data, -1)), ref(bo), host) == -3
    # precedence: a null pointer before a size error, a size error before a null input array
    assert _call(plan, ref(bi), ref(_lib.TbBucklingIn(0, None, -1)), ref(bo), host) == -1
    nx = _lib.TbBatchIn.from_buffer_copy(bi)
    nx.joint_xyz = None
    assert _call(plan, ref(nx), ref(_lib.TbBucklingIn(0, ax.ctypes.data, plan.M)), ref(bo), host) == -3
    assert _call(plan, ref(nx), ref(bki), ref(bo), host) == -1
    bad = _lib.TbBatchIn.from_buffer_copy(bi)
    bad.batch = -1
    assert _call(plan, ref(bad), ref(bki), ref(bo), host) == -3
    gene = np.zeros((B, plan.M), np.int32)             # a gene batch without a type table
    gb = _lib.TbBatchIn.from_buffer_copy(bi)
    gb.member_aed, gb.gene, gb.gene_stride, gb.type_table, gb.n_type = None, gene.ctypes.data, plan.M, None, 0
    assert _call(plan, ref(gb), ref(bki), ref(bo), host) == -1
    empty = _lib.TbBatchIn.from_buffer_copy(bi)        # an empty batch is a no-op once the arguments are valid
    empty.batch = 0
    assert _call(plan, ref(empty), ref(bki), ref(bo), host) in (0, _lib.TB_ERR_NO_DEVICE)


@pytest.mark.parametrize("host", [False, True], ids=["device", "host"])
def test_bar942_is_too_large(host):
    plan, joints, aed = _plan_and_inputs("bar-942_input_0")
    assert plan.n > 160
    keep = []
    bi = plan._batch_in(1, joints, aed, None, None, np.zeros(plan.N), keep)
    ax = np.zeros(plan.M)
    fac, info = np.zeros((1, 6)), np.zeros(1, np.int32)
    bo = _lib.TbBucklingOut(fac.ctypes.data, None, info.ctypes.data)
    bki = _lib.TbBucklingIn(6, ax.ctypes.data, 0)
    assert _call(plan, C.byref(bi), C.byref(bki), C.byref(bo), host) == _lib.TB_ERR_TOO_LARGE
    nx = _lib.TbBatchIn.from_buffer_copy(bi)           # (before the null-input check, as tb_modes)
    nx.joint_xyz = None
    assert _call(plan, C.byref(nx), C.byref(bki), C.byref(bo), host) == _lib.TB_ERR_TOO_LARGE
    with pytest.raises(_lib.TrussLibError) as e:
        plan.buckling_host(1, joints, ax, aed=aed, n_modes=6)
    assert e.value.code == _lib.TB_ERR_TOO_LARGE


@pytest.mark.skipif(_has_cuda(), reason="only meaningful on a machine without a GPU")
def test_no_device():
    plan, joints, aed = _plan_and_inputs()
    with pytest.raises(_lib.NoCudaDeviceError):
        plan.buckling_host(3, joints, np.zeros(plan.M), aed=aed, n_modes=6)
    keep = []
    bi = plan._batch_in(2, joints, aed, None, None, np.zeros(plan.N), keep)
    ax = np.zeros(plan.M)
    fac, info = np.zeros((2, 6)), np.zeros(2, np.int32)
    bo = _lib.TbBucklingOut(fac.ctypes.data, None, info.ctypes.data)
    assert _call(plan, C.byref(bi), C.byref(_lib.TbBucklingIn(6, ax.ctypes.data, 0)), C.byref(bo), False) == \
        _lib.TB_ERR_NO_DEVICE
    from python_stable_3d_truss_analysis_b200.batch import BucklingBatch
    from python_stable_3d_truss_analysis_b200.truss import Truss
    t = Truss(3).LoadFromJSON(data=H.load_json("ref_data/bar-72_input_0.json"))
    with pytest.raises(_lib.NoCudaDeviceError):
        t.SolveBuckling(6)
    with pytest.raises(Exception):
        t.GetBucklingFactors()
    with pytest.raises(_lib.NoCudaDeviceError):
        BucklingBatch(t, aed=aed[None], nMode=6)


def test_python_arguments():
    plan, joints, aed = _plan_and_inputs()
    with pytest.raises(ValueError):
        plan.buckling_host(2, joints, np.zeros(plan.M + 1), aed=aed)              # neither [M] nor [B, M]
    with pytest.raises(ValueError):
        plan.buckling_host(3, joints, np.zeros(2 * plan.M), aed=aed, axial_stride=plan.M)   # too short for 3 rows
    with pytest.raises(ValueError):
        plan.buckling_host(2, joints, np.zeros(2 * plan.M), aed=aed, axial_stride=-1)
    from python_stable_3d_truss_analysis_b200.batch import BucklingBatch
    from python_stable_3d_truss_analysis_b200.truss import Truss
    t = Truss(3).LoadFromJSON(data=H.load_json("ref_data/bar-72_input_0.json"))
    with pytest.raises(ValueError):
        BucklingBatch(t)                               # neither aed nor genes
    with pytest.raises(ValueError):
        BucklingBatch(t, aed=aed[None], genes=np.zeros((1, plan.M), np.int32))
