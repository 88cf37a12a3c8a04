"""Reverse mode of linear buckling without a GPU: the numpy load-factor gradients (oracle/buckling_adjoint.py
factor_grad) against five-point central differences of the lowest load factor with the member forces held fixed, the
chain through the static solve's adjoint (oracle/adjoint.py) against central differences of solve -> buckling, the
braced column's closed forms, the identities that follow from the homogeneity and invariances of K and K_G, and the
argument checks of tb_buckling_adjoint and autograd.buckling.

The finite differences evaluate the lowest factor through a vectorised assembly of K_ff and K_G,ff
(``lowest_factor``), which test_fast_matrices_equal_the_oracle checks against oracle/buckling.py on every fixture: the
oracle's per-member Python loops would take hours over every coordinate of bar-120."""
import ctypes as C
import functools

import numpy as np
import pytest
import scipy.linalg as sl

from oracle import adjoint as oadj
from oracle import buckling as bk
from oracle import buckling_adjoint as badj
from oracle import modal
from oracle import truss_oracle as orc
from python_stable_3d_truss_analysis_b200 import _lib
from tests import helpers as H
from tests.test_buckling_cpu import axial_of, braced_column, fixtures

TOL_FD = 1e-6
TOL_ID = 1e-11
CLEAR = 1e-6         # nu < -CLEAR max|nu|: a clearly critical mode (as tests/test_gpu_buckling.py)
FD_REL = 1e-4        # relative finite-difference step


def _has_cuda():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def cases():
    """(name, dim, joints, support, conn, aed, force): both braced columns and every fixture of test_buckling_cpu."""
    out = [(f"braced-column-{d}d", d) + braced_column(d) for d in (2, 3)]
    for name, dim, data in fixtures():
        out.append((name, dim) + tuple(orc.arrays_from_json(data, dim)))
    return out


CASES = {c[0]: c[1:] for c in cases()}


def matrices(dim, joints, support, conn, aed, axial):
    """(K_ff, K_G,ff) assembled vectorised over the members: oracle/buckling.py's forms."""
    conn = np.asarray(conn).astype(np.int64).reshape(-1, 2)
    M = conn.shape[0]
    d = joints[conn[:, 1]] - joints[conn[:, 0]]
    L = np.sqrt((d * d).sum(axis=1))
    c = d / L[:, None]
    cc = c[:, :, None] * c[:, None, :]
    kb = (aed[:, 1] * aed[:, 0] / L)[:, None, None] * cc
    gb = (np.asarray(axial, dtype=np.float64) / L)[:, None, None] * (np.eye(dim)[None] - cc)
    dofs = (conn[:, :, None] * dim + np.arange(dim)[None, None, :]).reshape(M, 2 * dim)
    sgn = np.kron(np.array([[1.0, -1.0], [-1.0, 1.0]]), np.ones((dim, dim)))
    N = joints.shape[0] * dim
    out = []
    for blk in (kb, gb):
        A = np.zeros((N, N))
        np.add.at(A, (dofs[:, :, None], dofs[:, None, :]), np.tile(blk, (1, 2, 2)) * sgn[None])
        out.append(A)
    mask = orc.free_mask(dim, support)
    return out[0][np.ix_(mask, mask)], out[1][np.ix_(mask, mask)]


def lowest_factor(dim, joints, support, conn, aed, axial):
    K, KG = matrices(dim, joints, support, conn, aed, axial)
    return -1.0 / sl.eigh(KG, K, eigvals_only=True, subset_by_index=[0, 0])[0]


def fd(f, x0, scale):
    """Five-point central differences of f at x0 with steps FD_REL * scale."""
    out = np.empty_like(x0)
    for i in range(x0.size):
        h = FD_REL * scale[i]
        e = np.zeros_like(x0)
        e[i] = h
        out[i] = (8.0 * (f(x0 + e) - f(x0 - e)) - (f(x0 + 2 * e) - f(x0 - 2 * e))) / (12.0 * h)
    return out


def assert_close(got, want, tol, what):
    err = orc.normwise_err(np.ravel(got), np.ravel(want))
    assert err <= tol, f"{what}: norm-wise err {err:.3e} > {tol:g}"


@functools.lru_cache(maxsize=None)
def forward(name):
    """(dim, joints, support, conn, aed, force, axial, oracle buckling result)"""
    dim, joints, support, conn, aed, force = CASES[name]
    ax = axial_of(dim, joints, support, conn, aed, force)
    return dim, joints, support, conn, aed, force, ax, bk.buckling(dim, joints, support, conn, aed, ax)


def simple_lowest(r):
    nu = r["nu"]
    lo = nu < -CLEAR * np.abs(nu).max()
    return bool(lo[0]) and len(modal.clusters(r["factor_all"][lo], 1e-6)[0]) == 1


FD_NAMES = [n for n in CASES if simple_lowest(forward(n)[-1])]


def test_the_fd_cases():
    """Every fixture but bar-72_input_0 (an exactly repeated lowest pair) and the 3D column has a simple lowest factor."""
    assert set(CASES) - set(FD_NAMES) == {"bar-72_input_0", "braced-column-3d"}


@pytest.mark.parametrize("name", list(CASES))
def test_fast_matrices_equal_the_oracle(name):
    dim, joints, support, conn, aed, force, ax, r = forward(name)
    K, KG = matrices(dim, joints, support, conn, aed, ax)
    assert np.abs(K - r["K_ff"]).max() <= 1e-13 * np.abs(r["K_ff"]).max()
    assert np.abs(KG - r["K_G_ff"]).max() <= 1e-13 * np.abs(r["K_G_ff"]).max()
    assert np.abs(orc.solve_closed_form(dim, joints, support, conn, aed, force)["axial"] - ax).max() <= \
        1e-11 * np.abs(ax).max()


@pytest.mark.parametrize("name", FD_NAMES)
def test_factor_grad_matches_finite_differences(name):
    """N held fixed: dlambda_0/d(xyz, a, E, N) against differences of the lowest factor."""
    dim, joints, support, conn, aed, force, ax, r = forward(name)
    gx, ga, gn = badj.factor_grad(dim, joints, support, conn, aed, ax, r["factor"][:1], r["modes"][:1], [1.0])
    nx, na = joints.size, len(conn)
    x0 = np.concatenate([joints.ravel(), aed[:, 0], aed[:, 1], ax])
    scale = np.concatenate([np.full(nx, np.ptp(joints, axis=0).max()), aed[:, 0], aed[:, 1],   # (N: forces near 0
                            np.full(na, np.abs(ax).mean())])                                 # are rounding)

    def f(x):
        a = np.stack([x[nx:nx + na], x[nx + na:nx + 2 * na], aed[:, 2]], 1)
        return lowest_factor(dim, x[:nx].reshape(joints.shape), support, conn, a, x[nx + 2 * na:])

    want = fd(f, x0, scale)
    assert_close(gx, want[:nx], TOL_FD, f"{name} xyz")
    assert_close(ga[:, :2].T, want[nx:nx + 2 * na], TOL_FD, f"{name} (a, E)")
    assert_close(gn, want[nx + 2 * na:], TOL_FD, f"{name} N")
    assert not ga[:, 2].any()


def total_grad(dim, joints, support, conn, aed, force, ax, r, g):
    """dL/d(xyz, aed, force) through the static solve: factor_grad, then oracle/adjoint.py with g_axial = dL/dN."""
    gx, ga, gn = badj.factor_grad(dim, joints, support, conn, aed, ax, r["factor"], r["modes"], g)
    s = oadj.adjoint(dim, joints, support, conn, aed, force, g_axial=gn)
    return gx + s["joint_xyz"], ga + s["member_aed"], s["force"], (gx, ga, gn)


@pytest.mark.parametrize("name", [n for n in FD_NAMES if n in ("braced-column-2d", "bar-6_input_0", "bar-10_input_0",
                                                              "bar-25_input_0", "bar-47_input_0", "bar-72_input_1",
                                                              "cube-7_case_1")])
def test_chain_matches_finite_differences_of_solve_then_buckling(name):
    dim, joints, support, conn, aed, force, ax, r = forward(name)
    k = len(r["factor"])
    g = np.zeros(k)
    g[0] = 1.0
    gx, ga, gf, _ = total_grad(dim, joints, support, conn, aed, force, ax, r, g)
    nx, na, nf = joints.size, len(conn), force.size
    x0 = np.concatenate([joints.ravel(), aed[:, 0], aed[:, 1], force])
    scale = np.concatenate([np.full(nx, np.ptp(joints, axis=0).max()), aed[:, 0], aed[:, 1],
                            np.full(nf, np.abs(force).max())])

    def f(x):
        j = x[:nx].reshape(joints.shape)
        a = np.stack([x[nx:nx + na], x[nx + na:nx + 2 * na], aed[:, 2]], 1)
        n = orc.solve_closed_form(dim, j, support, conn, a, x[nx + 2 * na:])["axial"]
        return lowest_factor(dim, j, support, conn, a, n)

    want = fd(f, x0, scale)
    mask = orc.free_mask(dim, support)
    assert_close(gx, want[:nx], TOL_FD, f"{name} xyz")
    assert_close(ga[:, :2].T, want[nx:nx + 2 * na], TOL_FD, f"{name} (a, E)")
    assert_close(gf[mask], want[nx + 2 * na:][mask], TOL_FD, f"{name} force")
    assert not gf[~mask].any() and np.abs(want[nx + 2 * na:][~mask]).max() <= 1e-9 * np.abs(gf).max()


@pytest.mark.parametrize("dim", [2, 3])
def test_braced_column_closed_forms(dim):
    """lambda = Es As L / (b P): dlambda/dAs = lambda / As, dlambda/dEs = lambda / Es, dlambda/dN_column = lambda / P
    (N = -P), the column's (a, E) gradient 0 and dlambda/dP = -lambda / P through the solve.  In 3D the lowest factor
    is a pair (one per brace), so the cotangent is 1 on both and each brace carries its own factor's gradient."""
    Es, As, L, b, P = 3.0e7, 0.25, 4.0, 3.0, 1.0e3
    joints, support, conn, aed, force = braced_column(dim, Es=Es, As=As, L=L, b=b, P=P)
    ax = axial_of(dim, joints, support, conn, aed, force)
    r = bk.buckling(dim, joints, support, conn, aed, ax)
    lam, npair = Es * As * L / (b * P), dim - 1
    g = np.zeros(len(r["factor"]))
    g[:npair] = 1.0
    gx_t, ga_t, gf, (gx, ga, gn) = total_grad(dim, joints, support, conn, aed, force, ax, r, g)
    for grads in (ga, ga_t):                                  # explicit, and through the solve (N does not change)
        assert grads[1:, 0] == pytest.approx(np.full(npair, lam / As), rel=1e-12)
        assert grads[1:, 1] == pytest.approx(np.full(npair, lam / Es), rel=1e-12)
        assert np.abs(grads[0, :2]).max() <= 1e-12 * lam / As
        assert not grads[:, 2].any()
    assert gn[0] == pytest.approx(npair * lam / P, rel=1e-12)
    if dim == 2:                                              # tension in the brace does not stiffen its own direction
        assert np.abs(gn[1]) <= 1e-12 * lam / P
    else:                                                     # ... but the other one: lambda^2 / (Es As) per brace
        assert gn[1:] == pytest.approx(np.full(2, lam * lam / (Es * As)), rel=1e-12)
    assert -gf[2 * dim - 1] == pytest.approx(-npair * lam / P, rel=1e-12)   # f_z(J1) = -P


def identities(dim, joints, support, conn, aed, force, ax, L, explicit, total):
    """The residuals of the exact identities of DESIGN.md section 12, each divided by |L|:
      sum E dL/dE = L, sum a dL/da = L           (explicit and total: K linear in a and E, N unchanged by their scale)
      sum N dL/dN = -L                            (explicit: lambda is homogeneous of degree -1 in N)
      sum x.dL/dx = 0, sum_J dL/dx_J = 0          (explicit and total: K, K_G ~ 1/s, N scale-free; translation)
      sum_J x_J x dL/dx_J = 0                     (3D, pins only: rotation; the total with the loads rotated
                                                  too: sum_J x_J x dL/dx_J + f_J x dL/df_J = 0)
      sum f.dL/df = -L                            (total: the loads scale N)
      dL/drho = 0"""
    gx, ga, gn = explicit
    tx, ta, tf = total
    r = [np.dot(aed[:, 1], ga[:, 1]) - L, np.dot(aed[:, 0], ga[:, 0]) - L, np.dot(ax, gn) + L,
         np.sum(joints * gx), np.abs(gx.sum(axis=0)).max(),
         np.dot(aed[:, 1], ta[:, 1]) - L, np.dot(aed[:, 0], ta[:, 0]) - L, np.sum(joints * tx),
         np.abs(tx.sum(axis=0)).max(), np.dot(force, tf) + L, np.abs(ga[:, 2]).max() + np.abs(ta[:, 2]).max()]
    if dim == 3 and set(np.unique(support)) <= {orc.NO, orc.PIN}:
        r += [np.abs(np.cross(joints, gx).sum(axis=0)).max(),
              np.abs(np.cross(joints, tx).sum(axis=0) + np.cross(force.reshape(-1, 3), tf.reshape(-1, 3)).sum(axis=0)).max()]
    return np.abs(np.array(r)) / abs(L)


def clear_cotangent(r, seed):
    """Positive cotangents (no cancellation in L) on the clearly critical factors, 0 on the others."""
    nu = r["nu"][:len(r["factor"])]
    g = np.random.default_rng(seed).uniform(0.5, 1.5, len(nu))
    return np.where(nu < -CLEAR * np.abs(r["nu"]).max(), g, 0.0)


@pytest.mark.parametrize("name", list(CASES))
def test_identities(name):
    dim, joints, support, conn, aed, force, ax, r = forward(name)
    g = clear_cotangent(r, 5)
    L = float(g @ np.where(g != 0.0, r["factor"], 0.0))
    tx, ta, tf, explicit = total_grad(dim, joints, support, conn, aed, force, ax, r, g)
    assert identities(dim, joints, support, conn, aed, force, ax, L, explicit, (tx, ta, tf)).max() <= TOL_ID


def test_infinite_factors_and_zero_cotangents_are_skipped():
    """A +inf factor (zero mode row) with any cotangent, and a zero cotangent on a finite factor, contribute nothing."""
    dim, joints, support, conn, aed, force, ax, r = forward("bar-10_input_0")
    fac = r["factor"]
    assert np.isinf(fac).any()
    g = np.where(np.isfinite(fac), 1.0, np.inf)
    want = badj.factor_grad(dim, joints, support, conn, aed, ax, fac[np.isfinite(fac)], r["modes"][np.isfinite(fac)],
                            np.ones(int(np.isfinite(fac).sum())))
    got = badj.factor_grad(dim, joints, support, conn, aed, ax, fac, r["modes"], g)
    for a, b in zip(got, want):
        assert np.array_equal(a, b)
    zero = badj.factor_grad(dim, joints, support, conn, aed, 0.0 * ax, np.full(len(fac), np.inf), 0.0 * r["modes"],
                            np.ones(len(fac)))
    assert all(not z.any() and np.all(np.isfinite(z)) for z in zero)


# ---- C ABI ---------------------------------------------------------------------------------------------------------
def _plan_and_inputs(name="bar-72_input_0"):
    data = H.load_json(f"ref_data/{name}.json")
    dim = H.dim_of(name)
    joints, support, conn, aed, _ = orc.arrays_from_json(data, dim)
    return _lib.Plan(dim, conn, support), joints, aed


def _buffers(plan, B, k):
    bufs = {"factor": np.zeros((B, k)), "modes": np.zeros((B, k, plan.N)), "info": np.zeros(B, np.int32),
            "g": np.ones((B, k)), "ax": np.zeros((B, plan.M)), "gx": np.zeros((B, plan.nJ, plan.dim)),
            "ga": np.zeros((B, plan.M, 3)), "gn": np.zeros((B, plan.M))}
    ai = _lib.TbModesAdjIn(bufs["factor"].ctypes.data, bufs["modes"].ctypes.data, bufs["info"].ctypes.data,
                           bufs["g"].ctypes.data)
    ao = _lib.TbBucklingAdjOut(bufs["gx"].ctypes.data, bufs["ga"].ctypes.data, bufs["gn"].ctypes.data)
    bki = _lib.TbBucklingIn(k, bufs["ax"].ctypes.data, plan.M)
    return bufs, bki, ai, ao


def _call(plan_h, bi, bki, ai, ao):
    return _lib.lib().tb_buckling_adjoint(plan_h, bi, bki, ai, ao, None)


def test_abi_structs_and_export():
    assert "tb_buckling_adjoint" in _lib.EXPORTS
    assert [f[0] for f in _lib.TbBucklingAdjOut._fields_] == ["joint_xyz", "member_aed", "axial"]


def test_argument_errors():
    plan, joints, aed = _plan_and_inputs()
    keep = []
    B, k = 2, 6
    bi = plan._batch_in(B, joints, aed, None, None, np.zeros(plan.N), keep)
    bi.force = None                                    # (not read)
    bufs, bki, ai, ao = _buffers(plan, B, k)
    ref = C.byref
    assert _call(None, ref(bi), ref(bki), ref(ai), ref(ao)) == -1
    assert _call(plan._h, None, ref(bki), ref(ai), ref(ao)) == -1
    assert _call(plan._h, ref(bi), None, ref(ai), ref(ao)) == -1
    assert _call(plan._h, ref(bi), ref(bki), None, ref(ao)) == -1
    assert _call(plan._h, ref(bi), ref(bki), ref(ai), None) == -1
    assert _call(plan._h, ref(bi), ref(_lib.TbBucklingIn(k, None, plan.M)), ref(ai), ref(ao)) == -1   # axial
    for f in ("eigval", "modes", "info", "g_eigval"):  # every forward array and the cotangent are required
        bad = _lib.TbModesAdjIn.from_buffer_copy(ai)
        setattr(bad, f, None)
        assert _call(plan._h, ref(bi), ref(bki), ref(bad), ref(ao)) == -1, f
    for nm in (0, -1, plan.n + 1):
        assert _call(plan._h, ref(bi), ref(_lib.TbBucklingIn(nm, bufs["ax"].ctypes.data, plan.M)), ref(ai), ref(ao)) == -3
    assert _call(plan._h, ref(bi), ref(_lib.TbBucklingIn(k, bufs["ax"].ctypes.data, -1)), ref(ai), ref(ao)) == -3
    # precedence: a null pointer before a size error, a size error before a null input array
    assert _call(plan._h, ref(bi), ref(_lib.TbBucklingIn(0, None, -1)), ref(ai), ref(ao)) == -1
    nx = _lib.TbBatchIn.from_buffer_copy(bi)
    nx.joint_xyz = None
    assert _call(plan._h, ref(nx), ref(_lib.TbBucklingIn(0, bufs["ax"].ctypes.data, plan.M)), ref(ai), ref(ao)) == -3
    assert _call(plan._h, ref(nx), ref(bki), ref(ai), ref(ao)) == -1
    neg = _lib.TbBatchIn.from_buffer_copy(bi)
    neg.batch = -1
    assert _call(plan._h, ref(neg), ref(bki), ref(ai), ref(ao)) == -3
    table = np.array([[1.0, 1e7, 0.1]])                 # a gene / type-table batch has no member gradient
    gb = plan._batch_in(B, joints, None, np.zeros((B, plan.M), np.int32), table, np.zeros(plan.N), keep)
    assert _call(plan._h, ref(gb), ref(bki), ref(ai), ref(ao)) == -1
    empty = _lib.TbBatchIn.from_buffer_copy(bi)        # an empty batch is a no-op once the arguments are valid
    empty.batch = 0
    assert _call(plan._h, ref(empty), ref(bki), ref(ai), ref(ao)) in (0, _lib.TB_ERR_NO_DEVICE)
    skip = _lib.TbBucklingAdjOut(None, None, None)      # every output may be skipped
    assert _call(plan._h, ref(empty), ref(bki), ref(ai), ref(skip)) in (0, _lib.TB_ERR_NO_DEVICE)


def test_bar942_is_too_large():
    plan, joints, aed = _plan_and_inputs("bar-942_input_0")
    assert plan.n > 160
    keep = []
    bi = plan._batch_in(1, joints, aed, None, None, np.zeros(plan.N), keep)
    bufs, bki, ai, ao = _buffers(plan, 1, 6)
    assert _call(plan._h, C.byref(bi), C.byref(bki), C.byref(ai), C.byref(ao)) == _lib.TB_ERR_TOO_LARGE
    nx = _lib.TbBatchIn.from_buffer_copy(bi)           # (before the null-input check, as tb_buckling)
    nx.joint_xyz = None
    assert _call(plan._h, C.byref(nx), C.byref(bki), C.byref(ai), C.byref(ao)) == _lib.TB_ERR_TOO_LARGE


@pytest.mark.skipif(_has_cuda(), reason="only meaningful on a machine without a GPU")
def test_no_device():
    plan, joints, aed = _plan_and_inputs()
    keep = []
    bi = plan._batch_in(3, joints, aed, None, None, np.zeros(plan.N), keep)
    bufs, bki, ai, ao = _buffers(plan, 3, 6)
    assert _call(plan._h, C.byref(bi), C.byref(bki), C.byref(ai), C.byref(ao)) == _lib.TB_ERR_NO_DEVICE
    shared = _lib.TbBucklingIn(6, bufs["ax"].ctypes.data, 0)
    assert _call(plan._h, C.byref(bi), C.byref(shared), C.byref(ai), C.byref(ao)) == _lib.TB_ERR_NO_DEVICE


def test_autograd_argument_types():
    """dtype, device and the choice of axial or force are checked before anything runs (shapes and batch sizes:
    tests/test_gpu_buckling_adjoint.py, which has CUDA tensors to pass)."""
    torch = pytest.importorskip("torch")
    from python_stable_3d_truss_analysis_b200 import autograd
    from python_stable_3d_truss_analysis_b200.truss import Truss

    t = Truss(3).LoadFromJSON(data=H.load_json("ref_data/bar-72_input_0.json"))
    joints, _, _, aed, force = t._pack()
    with pytest.raises(TypeError):
        autograd.buckling(t, xyz=torch.tensor(joints, dtype=torch.float32))
    with pytest.raises(TypeError):
        autograd.buckling(t, aed=torch.tensor(aed, dtype=torch.float64))           # a CPU tensor
    with pytest.raises(TypeError):
        autograd.buckling(t, axial=torch.zeros(t.nMember, dtype=torch.float64))   # a CPU tensor
    with pytest.raises(TypeError):
        autograd.buckling(t, force=torch.tensor(force, dtype=torch.float64))       # a CPU tensor
    with pytest.raises(ValueError):                                                # member forces or loads, not both
        autograd.buckling(t, axial=torch.zeros(t.nMember, dtype=torch.float64),
                          force=torch.tensor(force, dtype=torch.float64))
