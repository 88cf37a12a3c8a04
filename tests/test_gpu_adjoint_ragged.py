"""Reverse mode of ragged batches on the GPU (tb_adjoint_ragged, autograd.solve_ragged): per truss against the numpy
adjoint of oracle/adjoint.py (1e-9 norm-wise per field), bit for bit against the uniform adjoint of the same trusses,
batch independence, the kernels that ran, failed trusses among good ones, gradcheck and the compliance identity on 65 536
trusses generated on the device."""
import json

import numpy as np
import pytest

from oracle import adjoint as adj
from oracle import truss_oracle as orc
from python_stable_3d_truss_analysis_b200 import _lib
from tests import helpers as H
from tests.test_gpu_adjoint import FIELDS, assert_grads_close, device_adjoint, random_grads

pytestmark = pytest.mark.gpu

WARPS_MAX = 8            # the ragged adjoint kernels run at most 8 warps (trusses) per CTA
SMS = 148


def _torch():
    import torch
    return torch


def fixture(name):
    """(dim, joints, support, conn, aed, force) of a shipped fixture, a cube-7 case or a live_random entry."""
    if name.startswith("cube-7"):
        data = json.load(open(f"{H.GOLDEN}/ref_generate/{name}.json"))
        return (3,) + tuple(orc.arrays_from_json(data, 3))
    if name.startswith("random"):
        c = H.load_json("live_random.json")[int(name[6:])]
        return (c["dim"],) + tuple(orc.arrays_from_json(c["data"], c["dim"]))
    dim = H.dim_of(name + "_")
    return (dim,) + tuple(orc.arrays_from_json(json.load(open(f"{H.GOLDEN}/ref_data/{name}_input_0.json")), dim))


def pack(trusses):
    """Packed numpy arrays (tb_ragged_in layout) of [(joints, support, conn, aed, force)]."""
    nj = [len(t[0]) for t in trusses]
    nm = [len(t[2]) for t in trusses]
    jo, mo = np.zeros(len(trusses) + 1, np.int64), np.zeros(len(trusses) + 1, np.int64)
    jo[1:], mo[1:] = np.cumsum(nj), np.cumsum(nm)
    cat = lambda i, dt: np.concatenate([np.asarray(t[i], dt).reshape(-1) for t in trusses])  # noqa: E731
    return {"joint_off": jo, "member_off": mo, "xyz": cat(0, np.float64), "support": cat(1, np.uint8),
            "conn": cat(2, np.int32), "aed": cat(3, np.float64), "force": cat(4, np.float64)}


def ragged_grads(rng, p, dim):
    SJ, SM, B = int(p["joint_off"][-1]), int(p["member_off"][-1]), len(p["joint_off"]) - 1
    return {"u": rng.standard_normal(SJ * dim), "ext": rng.standard_normal(SJ * dim), "axial": rng.standard_normal(SM),
            "weight": rng.standard_normal(B)}


def ragged_adjoint(dim, p, grads, max_joint=None, max_member=None):
    """Forward (tb_solve_ragged) and reverse (tb_adjoint_ragged) of packed numpy arrays; numpy results."""
    torch = _torch()
    dev = torch.device("cuda:0")
    d = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in p.items()}
    fwd = _lib.solve_ragged_device(dim, d, max_joint=max_joint, max_member=max_member)
    SJ, SM, B = int(p["joint_off"][-1]), int(p["member_off"][-1]), len(p["joint_off"]) - 1
    f64 = dict(dtype=torch.float64, device=dev)
    res = {"joint_xyz": torch.full((SJ * dim,), np.nan, **f64), "member_aed": torch.full((SM * 3,), np.nan, **f64),
           "force": torch.full((SJ * dim,), np.nan, **f64), "info": torch.full((B,), 99, dtype=torch.int32, device=dev)}
    g = {k: torch.from_numpy(v).to(dev) for k, v in grads.items()}
    _lib.adjoint_ragged_device(dim, d, fwd["u"], g, res, max_joint=max_joint, max_member=max_member)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in fwd.items()}, {k: v.cpu().numpy() for k, v in res.items()}


def truss_slices(p, b, dim):
    j0, j1, m0, m1 = (int(x) for x in (p["joint_off"][b], p["joint_off"][b + 1], p["member_off"][b], p["member_off"][b + 1]))
    return slice(j0 * dim, j1 * dim), slice(m0, m1), slice(3 * m0, 3 * m1)


def per_truss(res, p, b, dim):
    """The gradients of truss b shaped as the oracle returns them."""
    sj, _, sm3 = truss_slices(p, b, dim)
    return {"joint_xyz": res["joint_xyz"][sj].reshape(-1, dim), "member_aed": res["member_aed"][sm3].reshape(-1, 3),
            "force": res["force"][sj]}


def per_truss_grads(grads, p, b, dim):
    sj, sm, _ = truss_slices(p, b, dim)
    return dict(g_u=grads["u"][sj], g_ext=grads["ext"][sj], g_axial=grads["axial"][sm], g_w=float(grads["weight"][b]))


# Trusses whose d/dE column is a near-total cancellation under the cotangents of these tests: the column is
# (A/L)(c.du) q with q = N^ - c.d(lambda), and on live_random 19 (3D, 4 joints) its terms are ~1e6 times its value, so
# rounding alone puts its error near 1e-7 of its own size in any summation order.  Only that column of these trusses is
# measured against the size of its terms; every other column and field is checked as assert_grads_close does.
E_COLUMN_CANCELS = {"random19"}


def assert_e_column_close_to_its_terms(got, want, dim, truss, g, what, tol=1e-9):
    joints, support, conn, aed, _ = truss
    mask = orc.free_mask(dim, support)
    J = lambda v: np.asarray(v).reshape(-1, dim)                     # noqa: E731
    d = joints[conn[:, 1]] - joints[conn[:, 0]]
    L = np.linalg.norm(d, axis=1)
    c = d / L[:, None]
    delta = lambda v: (c * (J(v)[conn[:, 1]] - J(v)[conn[:, 0]])).sum(axis=1)   # noqa: E731
    q_terms = np.maximum(np.abs(g["g_axial"] + delta(np.where(mask, 0.0, g["g_ext"]))), np.abs(delta(want["lam"])))
    terms = aed[:, 0] / L * np.abs(delta(want["u"])) * q_terms
    scale = max(np.abs(want["member_aed"][:, 1]).max(), terms.max())
    err = np.abs(got["member_aed"][:, 1] - want["member_aed"][:, 1]).max() / scale
    assert err <= 100 * tol, f"{what} d/de: err {err:.3e} relative to its terms"


def check_vs_oracle(dim, names, trusses, seed):
    """Every truss of these batches has a reference solution (the shipped fixtures, the cube-7 cases, live_random), so
    every one must solve (info 0) and match the oracle."""
    p = pack(trusses)
    grads = ragged_grads(np.random.default_rng(seed), p, dim)
    _, got = ragged_adjoint(dim, p, grads)
    failed = [(names[b], int(got["info"][b])) for b in np.flatnonzero(got["info"])]
    assert not failed, failed
    for b, (name, t) in enumerate(zip(names, trusses)):
        g = {k: [v] for k, v in per_truss(got, p, b, dim).items()}
        tg = per_truss_grads(grads, p, b, dim)
        want = adj.adjoint(dim, *t, **tg)
        if name not in E_COLUMN_CANCELS:
            assert_grads_close(g, want, 0, what=f"{name} at {b}")
            continue
        for k in FIELDS:                                               # assert_grads_close without the e column
            assert orc.normwise_err(g[k][0], want[k]) <= 1e-9, (name, k)
        for col in (0, 2):
            assert orc.normwise_err(g["member_aed"][0][:, col], want["member_aed"][:, col]) <= 1e-7, (name, col)
        assert_e_column_close_to_its_terms({k: v[0] for k, v in g.items()}, want, dim, t, tg, what=f"{name} at {b}")


def test_mixed_3d_batch_vs_oracle():
    randoms = [f"random{i}" for i, c in enumerate(H.load_json("live_random.json")) if c["dim"] == 3]
    names = ["bar-6", "bar-25", "bar-72", "bar-120"] + [c[0] for c in H.cube7_shipped()] + randoms
    rng = np.random.default_rng(1)
    names = [names[i] for i in rng.permutation(len(names))]
    check_vs_oracle(3, names, [fixture(n)[1:] for n in names], seed=2)


def test_mixed_2d_batch_vs_oracle():
    randoms = [f"random{i}" for i, c in enumerate(H.load_json("live_random.json")) if c["dim"] == 2]
    names = ["bar-10", "bar-47"] + randoms
    rng = np.random.default_rng(3)
    names = [names[i] for i in rng.permutation(len(names))]
    check_vs_oracle(2, names, [fixture(n)[1:] for n in names], seed=4)


def perturbed_copies(name, B=5, seed=2):
    dim, joints, support, conn, aed, force = fixture(name)
    rng = np.random.default_rng(seed)
    xyzb = joints[None] + rng.normal(0, 0.01, size=(B,) + joints.shape)
    aedb = aed[None] * rng.uniform(0.5, 2.0, size=(B, aed.shape[0], 1))
    F = force.reshape(1, -1) * rng.uniform(0.5, 2.0, size=(B, 1))
    return dim, support, conn, xyzb, aedb, F


@pytest.mark.parametrize("name", ["bar-72", "bar-25", "bar-10", "bar-47", "bar-120"])
def test_bit_identical_to_the_uniform_adjoint(name):
    """The same trusses through Plan.adjoint_device on the fused path and as a ragged batch: the same member bodies, the
    same summation orders and the same solve kernel give the same bits (bar-120 solves on k_small under ragged sizing)."""
    dim, support, conn, xyzb, aedb, F = perturbed_copies(name)
    B = xyzb.shape[0]
    plan = _lib.Plan(dim, conn, support)
    assert plan.path == 0
    rng = np.random.default_rng(7)
    grads = random_grads(rng, B, plan.N, plan.M)
    _, uni = device_adjoint(plan, xyzb, aedb, F, grads)
    p = pack([(xyzb[b], support, conn, aedb[b], F[b]) for b in range(B)])
    rg = {k: np.ascontiguousarray(v.reshape(-1)) for k, v in grads.items()}
    _, rag = ragged_adjoint(dim, p, rg)
    assert not uni["info"].any() and np.array_equal(uni["info"], rag["info"])
    for b in range(B):
        g = per_truss(rag, p, b, dim)
        for k in FIELDS:
            want = uni[k][b].reshape(g[k].shape)
            if name == "bar-120":
                assert orc.normwise_err(g[k], want) <= 1e-9, (k, b)
            else:
                assert np.array_equal(g[k], want), (k, b)


def cube7_batch(n, seed):
    trusses = [fixture(c[0])[1:] for c in H.cube7_shipped()]
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        joints, support, conn, aed, force = trusses[i % len(trusses)]
        out.append((joints + rng.normal(0.0, 0.5, size=joints.shape), support, conn,
                    aed * rng.uniform(0.5, 2.0, size=(aed.shape[0], 1)), force))
    return out


def test_deterministic_and_batch_independent():
    trusses = cube7_batch(2 * WARPS_MAX * SMS + 3, seed=5)
    p = pack(trusses)
    maxj = int(np.diff(p["joint_off"]).max())
    maxm = int(np.diff(p["member_off"]).max())
    grads = ragged_grads(np.random.default_rng(6), p, 3)
    _, one = ragged_adjoint(3, p, grads, maxj, maxm)
    _, two = ragged_adjoint(3, p, grads, maxj, maxm)
    assert not one["info"].any()
    for k in FIELDS:
        assert np.array_equal(one[k], two[k]), k
    for b in (0, 7, 1000, len(trusses) - 1):
        gb = {k: v[truss_slices(p, b, 3)[0 if k in ("u", "ext") else 1]] if k != "weight" else v[b:b + 1]
              for k, v in grads.items()}
        for pos in (0, 2):                                          # alone, and at another position
            others = [trusses[(b + 1) % len(trusses)], trusses[(b + 2) % len(trusses)]][:pos]
            q = pack(others + [trusses[b]])
            qg = ragged_grads(np.random.default_rng(8), q, 3)
            sj, sm, _ = truss_slices(q, pos, 3)
            for k in ("u", "ext"):
                qg[k][sj] = gb[k]
            qg["axial"][sm] = gb["axial"]
            qg["weight"][pos] = gb["weight"][0]
            _, single = ragged_adjoint(3, q, qg, maxj, maxm)
            got, want = per_truss(single, q, pos, 3), per_truss(one, p, b, 3)
            for k in FIELDS:
                assert np.array_equal(got[k], want[k]), (k, b, pos)


def _kernels(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [ev.name for ev in prof.events()]
    return {k for k in ("k_adj_rhs_ragged", "k_sens_ragged", "k_dense16", "k_small") if any(k in n for n in names)}


@pytest.mark.parametrize("B", [1, WARPS_MAX + 1, 8 * WARPS_MAX])
def test_kernels_that_ran(B):
    p = pack(cube7_batch(B, seed=B))
    grads = ragged_grads(np.random.default_rng(B), p, 3)
    ran = _kernels(lambda: ragged_adjoint(3, p, grads))
    assert {"k_adj_rhs_ragged", "k_dense16", "k_sens_ragged"} <= ran and "k_small" not in ran, ran
    # bar-120 under ragged sizing (d * max_joint = 147) no longer fits the warp kernel: the CTA-per-truss fallback
    names = (["bar-120"] + [c[0] for c in H.cube7_shipped()] * B)[:B]
    q = pack([fixture(n)[1:] for n in names])
    qg = ragged_grads(np.random.default_rng(B + 1), q, 3)
    ran = _kernels(lambda: ragged_adjoint(3, q, qg))
    assert {"k_adj_rhs_ragged", "k_small", "k_sens_ragged"} <= ran and "k_dense16" not in ran, ran
    _, got = ragged_adjoint(3, q, qg)
    assert not got["info"].any()
    want = adj.adjoint(3, *fixture(names[0])[1:], **per_truss_grads(qg, q, 0, 3))
    assert_grads_close({k: [v] for k, v in per_truss(got, q, 0, 3).items()}, want, 0, what="bar-120 on k_small")


def failing_trusses():
    """(expected status, truss) of every failure class; each is a cube-7 case with one defect."""
    base = fixture(H.cube7_shipped()[0][0])[1:]
    out = []
    joints, support, conn, aed, force = (np.array(a, copy=True) for a in base)
    joints[conn[0, 1]] = joints[conn[0, 0]]                          # zero-length member
    out.append((-2, (joints, support, conn, aed, force)))
    joints, support, conn, aed, force = (np.array(a, copy=True) for a in base)
    aed[:, 1] = 0.0                                                   # no stiffness at all: singular K
    out.append((1, (joints, support, conn, aed, force)))
    out.append((-1, (np.array([[0.0, 0, 0], [1, 0, 0]]), np.array([1, 0], np.uint8), np.array([[0, 1]], np.int32),
                     np.array([[1.0, 1e7, 1.0]]), np.zeros(6))))      # counting rule
    joints, support, conn, aed, force = (np.array(a, copy=True) for a in base)
    support[3] = 9                                                    # not a support code
    out.append((-3, (joints, support, conn, aed, force)))
    joints, support, conn, aed, force = (np.array(a, copy=True) for a in base)
    conn[5, 1] = len(joints) + 1000                                   # joint id out of range
    conn[9, 0] = -3
    out.append((-4, (joints, support, conn, aed, force)))
    return out


def test_failed_trusses_among_good_ones():
    good = cube7_batch(3 * WARPS_MAX, seed=9)
    bad = failing_trusses()
    mixed, where = [], []
    for i, t in enumerate(good):                                       # failures interleaved: they share CTAs with good ones
        mixed.append(t)
        if i % 4 == 1 and bad:
            where.append((len(mixed), bad[0][0]))
            mixed.append(bad.pop(0)[1])
    p = pack(mixed)
    maxj = int(np.diff(p["joint_off"]).max())
    maxm = int(np.diff(p["member_off"]).max())
    grads = ragged_grads(np.random.default_rng(10), p, 3)
    _, got = ragged_adjoint(3, p, grads, maxj, maxm)
    bad_idx = [b for b, _ in where]
    for b, status in where:
        assert (got["info"][b] > 0) if status > 0 else got["info"][b] == status, (b, status, got["info"][b])
        g = per_truss(got, p, b, 3)
        for k in FIELDS:
            assert np.isfinite(g[k]).all() and not g[k].any(), (k, status)
    good_idx = [b for b in range(len(mixed)) if b not in bad_idx]
    assert not got["info"][good_idx].any()
    # the good neighbours are bit for bit their gradients in a batch without the failures
    q = pack([mixed[b] for b in good_idx])
    qg = {"weight": grads["weight"][good_idx]}
    for k, src in (("u", 0), ("ext", 0), ("axial", 1)):
        qg[k] = np.concatenate([grads[k][truss_slices(p, b, 3)[src]] for b in good_idx])
    _, clean = ragged_adjoint(3, q, qg, maxj, maxm)
    for i, b in enumerate(good_idx):
        c, g = per_truss(clean, q, i, 3), per_truss(got, p, b, 3)
        for k in FIELDS:
            assert np.array_equal(c[k], g[k]), (k, b)


def test_autograd_gradcheck():
    torch = _torch()
    from python_stable_3d_truss_analysis_b200 import autograd

    names = ["bar-6", "bar-25", "bar-6"]
    p = pack([fixture(n)[1:] for n in names])
    dev = torch.device("cuda:0")
    d = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in p.items()}
    x0, a0, f0 = d["xyz"].reshape(-1, 3), d["aed"].reshape(-1, 3), d["force"]
    ref = autograd.solve_ragged(d)
    assert not ref["info"].any()
    scale = {k: ref[k].abs().max() for k in ("u", "ext", "axial", "weight")}
    span = float(np.ptp(p["xyz"].reshape(-1, 3), axis=0).max())

    def fn(dx, sa, sf):                          # relative perturbations of every input; outputs O(1)
        out = autograd.solve_ragged(d, xyz=x0 + span * dx, aed=a0 * sa, force=f0 * sf)
        return tuple(out[k] / scale[k] for k in ("u", "ext", "axial", "weight"))

    args = (torch.zeros_like(x0, requires_grad=True), torch.ones_like(a0, requires_grad=True),
            torch.ones_like(f0, requires_grad=True))
    assert torch.autograd.gradcheck(fn, args, eps=1e-6, atol=1e-5, rtol=1e-3)
    # d(f.u)/df = u + K^-1 f = 2u (u and the loads' gradient vanish at supported DOFs)
    f = f0.clone().requires_grad_(True)
    out = autograd.solve_ragged(d, force=f)
    (f * out["u"]).sum().backward()
    assert orc.normwise_err(f.grad.cpu().numpy(), 2.0 * out["u"].detach().cpu().numpy()) <= 1e-12


def test_backward_refuses_a_topology_changed_in_place():
    """The topology tensors are saved for the backward pass: changing conn in place after the forward is an error, not
    silently wrong gradients."""
    torch = _torch()
    from python_stable_3d_truss_analysis_b200 import autograd

    p = pack([fixture(n)[1:] for n in ("bar-6", "bar-25")])
    dev = torch.device("cuda:0")
    d = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in p.items()}
    a = d["aed"].clone().requires_grad_(True)
    out = autograd.solve_ragged(d, aed=a)
    d["conn"].add_(0)                                                   # (same values, new version)
    with pytest.raises(RuntimeError, match="inplace"):
        out["u"].sum().backward()


def _per_truss_max(B, owner, values, keep):
    out = np.zeros(B)
    np.maximum.at(out, owner[keep], values[keep])
    return out


def test_identities_on_generated_cube7_batch():
    """65 536 cube-7 trusses generated on the device, solved and differentiated without leaving it, through three exact
    identities per solved truss.  L = sum f.u + sum over free DOFs of ext (ext = f there):
      dL/dA_m = -N_m^2 L_m / (E_m A_m^2)     (compliance; the ext term does not depend on the members),
      sum over joints of dL/dxyz = 0          (translation invariance: every member adds +G at joint 1, -G at joint 0),
      dL/df = 2u + 1 at free DOFs, 0 at supported ones."""
    torch = _torch()
    from python_stable_3d_truss_analysis_b200 import autograd
    from python_stable_3d_truss_analysis_b200 import generate as G

    B = 65536
    gen = G.GenerateRandomCubeTrussesOnDevice(B, seed=17, gridRange=(5, 5, 5), numCubeRange=(7, 7), asNumpy=False)
    x = gen["xyz"].reshape(-1, 3).clone().requires_grad_(True)
    a = gen["aed"].clone().requires_grad_(True)
    f = gen["force"].clone().requires_grad_(True)
    sup = gen["support"].to(torch.int64)[:, None]
    axis = torch.arange(3, device=sup.device)[None, :]
    free = (~((sup == 1) | (sup == 2 + axis))).reshape(-1).to(torch.float64)       # the support rule, per DOF
    out = autograd.solve_ragged(gen, xyz=x, aed=a, force=f)
    ((f * out["u"]).sum() + (free * out["ext"]).sum()).backward()
    info = out["info"].cpu().numpy()
    assert (info == 0).sum() >= B // 2, np.unique(info, return_counts=True)
    solved = info == 0
    jo, mo = gen["joint_off"].cpu().numpy(), gen["member_off"].cpu().numpy()
    xyz = gen["xyz"].cpu().numpy().reshape(-1, 3)
    conn = gen["conn"].cpu().numpy().reshape(-1, 2).astype(np.int64)
    aed = gen["aed"].cpu().numpy().reshape(-1, 3)
    # compliance identity per member
    N = out["axial"].detach().cpu().numpy()
    ga = a.grad.cpu().numpy().reshape(-1, 3)
    tm = np.repeat(np.arange(B), np.diff(mo))                        # truss of every member
    base = jo[tm]
    L = np.sqrt(((xyz[base + conn[:, 1]] - xyz[base + conn[:, 0]]) ** 2).sum(axis=1))
    want = -N ** 2 * L / (aed[:, 1] * aed[:, 0] ** 2)
    okm = solved[tm]
    worst, scale = _per_truss_max(B, tm, np.abs(ga[:, 0] - want), okm), _per_truss_max(B, tm, np.abs(want), okm)
    assert (worst[solved] <= 1e-9 * scale[solved]).all(), (worst[solved] / scale[solved]).max()
    # translation invariance per truss
    gx = x.grad.cpu().numpy()
    tj = np.repeat(np.arange(B), np.diff(jo))                        # truss of every joint
    tot = np.zeros((B, 3))
    np.add.at(tot, tj, gx)
    okj = solved[tj]
    gscale = _per_truss_max(B, tj, np.abs(gx).max(axis=1), okj)
    assert (np.abs(tot).max(axis=1)[solved] <= 1e-10 * gscale[solved]).all()
    # load gradient per truss
    td = np.repeat(tj, 3)
    u = out["u"].detach().cpu().numpy()
    want_f = 2.0 * u + free.cpu().numpy()
    okd = solved[td]
    worst = _per_truss_max(B, td, np.abs(f.grad.cpu().numpy() - want_f), okd)
    scale = _per_truss_max(B, td, np.abs(want_f), okd)
    assert (worst[solved] <= 1e-12 * scale[solved]).all(), (worst[solved] / scale[solved]).max()
    # failed trusses: zero gradients everywhere
    assert not ga[~okm].any() and not gx[~okj].any() and not f.grad.cpu().numpy()[~okd].any()
