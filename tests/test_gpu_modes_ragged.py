"""Modal analysis of ragged batches on the GPU (tb_modes_ragged / tb_modes_ragged_host / tb_modes_adjoint_ragged,
k_modes_ragged<DIM> and k_modes_sens_ragged<DIM>, autograd.modes_ragged): mixed batches against the numpy oracle, bit
identity with the uniform kernels on the plan of the same topology, invariance under position, neighbours, B, max_joint
and max_free, padding, failures among good trusses, a 65 536-truss generated batch, gradcheck and CUDA graphs."""
import json

import numpy as np
import pytest

from oracle import modal
from oracle import truss_oracle as orc
from python_stable_3d_truss_analysis_b200 import _lib
from tests import helpers as H
from tests.test_gpu_modes import check_against_oracle, joint_masses, uncut

pytestmark = pytest.mark.gpu


def _torch():
    import torch
    return torch


def fixture(name):
    """(dim, joints, support, conn, aed) of a shipped fixture, a cube-7 case or a live_random entry."""
    if name.startswith("cube-7"):
        data = json.load(open(f"{H.GOLDEN}/ref_generate/{name}.json"))
        return (3,) + tuple(orc.arrays_from_json(data, 3)[:4])
    if name.startswith("random"):
        c = H.load_json("live_random.json")[int(name[6:])]
        return (c["dim"],) + tuple(orc.arrays_from_json(c["data"], c["dim"])[:4])
    dim = H.dim_of(name + "_")
    return (dim,) + tuple(orc.arrays_from_json(json.load(open(f"{H.GOLDEN}/ref_data/{name}_input_0.json")), dim)[:4])


def names(dim):
    out = [n[:-8] for n, d, _, _ in H.shipped_cases() if d == dim and not n.startswith("bar-942")]
    if dim == 3:
        out += [c[0] for c in H.cube7_shipped()[:2]]
    out += [f"random{i}" for i, c in enumerate(H.load_json("live_random.json")) if c["dim"] == dim]
    out = list(dict.fromkeys(out))
    return [n for n in out if _lib.Plan(fixture(n)[0], fixture(n)[3], fixture(n)[2]).n <= 160]


def pack(trusses, jm=None):
    nj, nm = [len(t[0]) for t in trusses], [len(t[2]) for t in trusses]
    jo, mo = np.zeros(len(trusses) + 1, np.int64), np.zeros(len(trusses) + 1, np.int64)
    jo[1:], mo[1:] = np.cumsum(nj), np.cumsum(nm)
    cat = lambda i, dt: np.concatenate([np.asarray(t[i], dt).reshape(-1) for t in trusses])  # noqa: E731
    p = {"joint_off": jo, "member_off": mo, "xyz": cat(0, np.float64), "support": cat(1, np.uint8), "conn": cat(2, np.int32),
         "aed": cat(3, np.float64)}
    if jm is not None:
        p["jm"] = np.concatenate(jm)
    return p


def device(p):
    torch = _torch()
    return {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in p.items()}


def run(dim, p, k, consistent=False, jm=False, **kw):
    """Forward on the device, numpy results."""
    d = device(p)
    out = _lib.modes_ragged_device(dim, d, k, consistent=consistent, joint_mass=d.get("jm") if jm else None, **kw)
    return {key: v.cpu().numpy() for key, v in out.items()}


def block(out, p, b, dim, k):
    jo = p["joint_off"]
    return out["modes"][k * dim * jo[b]:k * dim * jo[b + 1]].reshape(k, -1)


@pytest.mark.parametrize("jm", [False, True], ids=["plain", "joint_mass"])
@pytest.mark.parametrize("consistent", [False, True], ids=["lumped", "consistent"])
@pytest.mark.parametrize("dim", [3, 2])
def test_mixed_batch_against_oracle(dim, consistent, jm):
    ns = names(dim)
    ts = [fixture(n)[1:] for n in ns]
    masses = [joint_masses(dim, t[0], t[2], t[3]) for t in ts] if jm else None
    p = pack(ts, masses)
    k = 6
    out = run(dim, p, k, consistent, jm)
    for b, (n, t) in enumerate(zip(ns, ts)):
        assert out["info"][b] == 0, n
        ref = modal.modes(dim, *t, consistent=consistent, joint_mass=masses[b] if jm else None)
        nb = int(ref["mask"].sum())
        assert out["n_free"][b] == nb
        q = min(k, nb)                                         # (check_against_oracle handles clusters cut by q)
        check_against_oracle(dim, *t, out["eigval"][b, :q], block(out, p, b, dim, k)[:q], consistent, masses[b] if jm else None)


def plan_outputs(dim, joints, support, conn, aeds, k, consistent, jm=None):
    """tb_modes / tb_modes_adjoint on the plan of one topology, numpy results; cotangents fixed by a seed."""
    torch = _torch()
    plan = _lib.Plan(dim, conn, support)
    B = len(aeds)
    xyz = torch.from_numpy(np.tile(joints.reshape(1, -1), (B, 1))).cuda()
    aed = torch.from_numpy(np.stack(aeds)).cuda()
    jmt = None if jm is None else torch.from_numpy(np.tile(jm, (B, 1))).cuda()
    out = {"modes": torch.empty(B, k, plan.N, dtype=torch.float64, device="cuda")}
    plan.modes_device(B, xyz, aed=aed, n_modes=k, consistent=consistent, joint_mass=jmt, out=out)
    g = torch.from_numpy(np.random.default_rng(7).standard_normal((B, k))).cuda()
    res = {"joint_xyz": torch.empty(B, plan.nJ, dim, dtype=torch.float64, device="cuda"),
           "member_aed": torch.empty(B, plan.M, 3, dtype=torch.float64, device="cuda"),
           "joint_mass": torch.empty(B, plan.nJ, dtype=torch.float64, device="cuda")}
    plan.modes_adjoint_device(B, xyz, aed, out, g, res, n_modes=k, consistent=consistent)
    return {**{key: v.cpu().numpy() for key, v in out.items()}, **{key: v.cpu().numpy() for key, v in res.items()},
            "g": g.cpu().numpy()}


def ragged_with_adjoint(dim, p, k, consistent, g, jm=False, **kw):
    torch = _torch()
    d = device(p)
    fwd = _lib.modes_ragged_device(dim, d, k, consistent=consistent, joint_mass=d.get("jm") if jm else None, **kw)
    SJ, SM = int(p["joint_off"][-1]), int(p["member_off"][-1])
    res = {"joint_xyz": torch.empty(SJ * dim, dtype=torch.float64, device="cuda"),
           "member_aed": torch.empty(SM * 3, dtype=torch.float64, device="cuda"),
           "joint_mass": torch.empty(SJ, dtype=torch.float64, device="cuda")}
    gt = torch.from_numpy(np.ascontiguousarray(g)).cuda()
    mkw = {key: v for key, v in kw.items() if key in ("max_joint", "max_member", "max_free")}
    _lib.modes_adjoint_ragged_device(dim, d, fwd, gt, res, consistent=consistent, **mkw)
    return {**{key: v.cpu().numpy() for key, v in fwd.items()}, **{key: v.cpu().numpy() for key, v in res.items()}}


@pytest.mark.parametrize("consistent", [False, True], ids=["lumped", "consistent"])
@pytest.mark.parametrize("name", names(3) + names(2))
def test_bit_identical_to_the_uniform_kernels(name, consistent):
    dim, joints, support, conn, aed = fixture(name)
    rng = np.random.default_rng(3)
    aeds = [aed * rng.uniform(0.7, 1.4, size=(len(aed), 1)) for _ in range(4)]
    jm = joint_masses(dim, joints, conn, aed)
    n = _lib.Plan(dim, conn, support).n
    k = min(6, n)
    want = plan_outputs(dim, joints, support, conn, aeds, k, consistent, jm)
    p = pack([(joints, support, conn, a) for a in aeds], [jm] * len(aeds))
    got = ragged_with_adjoint(dim, p, k, consistent, want["g"], jm=True)
    assert np.array_equal(got["info"], want["info"])
    assert np.array_equal(got["eigval"], want["eigval"])
    nJ, M = len(joints), len(conn)
    for b in range(len(aeds)):
        assert np.array_equal(block(got, p, b, dim, k), want["modes"][b])
        assert np.array_equal(got["joint_xyz"][b * nJ * dim:(b + 1) * nJ * dim], want["joint_xyz"][b].reshape(-1))
        assert np.array_equal(got["member_aed"][b * M * 3:(b + 1) * M * 3], want["member_aed"][b].reshape(-1))
        assert np.array_equal(got["joint_mass"][b * nJ:(b + 1) * nJ], want["joint_mass"][b])


@pytest.mark.parametrize("consistent", [False, True], ids=["lumped", "consistent"])
def test_bits_do_not_depend_on_position_neighbours_or_launch(consistent):
    ns = [n for n in names(3) if not n.startswith("random")]
    ts = [fixture(n)[1:] for n in ns]
    k = 4
    ref = {}
    for i, t in enumerate(ts):                                 # each truss alone, default bound
        p = pack([t])
        ref[i] = (run(3, p, k, consistent), p)
    order = list(range(len(ts))) * 3
    np.random.default_rng(1).shuffle(order)
    p = pack([ts[i] for i in order])
    for kw in ({}, {"max_free": 160}, {"max_joint": int(np.diff(p["joint_off"]).max()) + 7}):
        out = run(3, p, k, consistent, **kw)
        for b, i in enumerate(order):
            o1, p1 = ref[i]
            assert out["info"][b] == o1["info"][0] == 0
            assert np.array_equal(out["eigval"][b], o1["eigval"][0])
            assert np.array_equal(block(out, p, b, 3, k), block(o1, p1, 0, 3, k))


def test_padding_n_free_and_an_all_pinned_truss():
    dim, joints, support, conn, aed = fixture("bar-6")
    j2, s2, c2, a2 = fixture("bar-72")[1:]
    pinned = (joints, np.full(len(joints), orc.PIN, np.uint8), conn, aed)
    p = pack([(joints, support, conn, aed), (j2, s2, c2, a2), pinned])
    k = 20
    n6 = _lib.Plan(dim, conn, support).n
    g = np.random.default_rng(2).standard_normal((3, k))
    out = ragged_with_adjoint(3, p, k, False, g)
    assert list(out["info"]) == [0, 0, 0]
    assert list(out["n_free"]) == [n6, 48, 0]
    assert np.all(out["eigval"][0, n6:] == 0) and np.all(out["eigval"][0, :n6] > 0)
    assert np.all(block(out, p, 0, 3, k)[n6:] == 0)
    assert np.all(out["eigval"][2] == 0) and np.all(block(out, p, 2, 3, k) == 0)
    alone = run(3, pack([(joints, support, conn, aed)]), n6)
    assert np.array_equal(out["eigval"][0, :n6], alone["eigval"][0])
    g2 = g.copy()
    g2[0, n6:] = np.random.default_rng(9).standard_normal(k - n6) * 1e3
    out2 = ragged_with_adjoint(3, p, k, False, g2)
    for key in ("joint_xyz", "member_aed", "joint_mass"):
        assert np.array_equal(out[key], out2[key])


def failing(dim):
    """(truss, reason) that fail a static guard, the free-DOF bound or the mass, for a 2D or 3D base fixture."""
    base = fixture("bar-6" if dim == 3 else "bar-10")[1:]
    joints, support, conn, aed = (np.array(x) for x in base)
    out = []
    sup = support.copy(); sup[:] = 0                                  # no support at all: counting rule
    out.append(((joints, sup, conn, aed), "not_stable"))
    j = joints.copy(); j[conn[0, 1]] = j[conn[0, 0]]                  # zero-length member
    out.append(((j, support, conn, aed), "zero_length"))
    s = support.copy(); s[0] = 7                                      # unknown support code
    out.append(((joints, s, conn, aed), "bad_support"))
    c = conn.copy(); c[1, 1] = len(joints) + 3                        # joint id out of range
    out.append(((joints, support, c, aed), "bad_index"))
    a = aed.copy(); a[:, 2] = 0.0                                     # no mass anywhere
    out.append(((joints, support, conn, a), "mass"))
    return out


@pytest.mark.parametrize("consistent", [False, True], ids=["lumped", "consistent"])
@pytest.mark.parametrize("dim", [3, 2])
def test_failures_among_good_trusses(dim, consistent):
    torch = _torch()
    good = [fixture(n)[1:] for n in names(dim)[:3]]
    bad = failing(dim)
    mixed = []
    for i, g in enumerate(good):
        mixed.append(g)
        mixed.append(bad[i % len(bad)][0])
    mixed += [b[0] for b in bad]
    p = pack(mixed)
    k = 3
    out = run(dim, p, k, consistent)
    alone = run(dim, pack(good), k, consistent)
    # statuses -1 ... -4 equal tb_solve_ragged's
    d = device(p)
    d["force"] = torch.zeros(int(p["joint_off"][-1]) * dim, dtype=torch.float64, device="cuda")
    static = _lib.solve_ragged_device(dim, d)["info"].cpu().numpy()
    for b, t in enumerate(mixed):
        if static[b] < 0:
            assert out["info"][b] == static[b], b
        if out["info"][b] != 0:
            assert np.all(out["eigval"][b] == 0) and np.all(block(out, p, b, dim, k) == 0) and out["n_free"][b] == 0
    pg = pack(good)
    for i in range(len(good)):
        assert np.array_equal(out["eigval"][2 * i], alone["eigval"][i])
        assert np.array_equal(block(out, p, 2 * i, dim, k), block(alone, pg, i, dim, k))
    reasons = {r: out["info"][2 * len(good) + j] for j, (_, r) in enumerate(bad)}
    assert reasons == {"not_stable": -1, "zero_length": -2, "bad_support": -3, "bad_index": -4, "mass": -5}
    # more free DOFs than the launch's bound
    small = fixture("bar-6" if dim == 3 else "bar-10")[1:]
    big = fixture("bar-72" if dim == 3 else "bar-47")[1:]
    p2 = pack([small, big])
    n_small = int(run(dim, pack([small]), 1)["n_free"][0])
    out2 = run(dim, p2, 1, consistent, max_free=n_small)
    assert out2["info"][0] == 0 and out2["info"][1] == -4


def test_mechanism_is_info_0_with_a_zero_eigenvalue():
    # a pyramid on four pins with one more bar standing on its apex: the bar's free end can swing sideways, yet the
    # counting rule holds (9 members + 12 restraints >= 18 DOFs)
    joints = np.array([[0, 0, 0], [1, 0, 0], [1, 1, 0], [0, 1, 0], [0.5, 0.5, 1.0], [0.5, 0.5, 2.0]], float)
    support = np.array([1, 1, 1, 1, 0, 0], np.uint8)
    conn = np.array([[0, 4], [1, 4], [2, 4], [3, 4], [4, 5], [0, 1], [1, 2], [2, 3], [3, 0]], np.int32)
    aed = np.tile([1.0, 1e4, 1.0], (len(conn), 1))
    p = pack([(joints, support, conn, aed)])
    out = run(3, p, 2)
    assert out["info"][0] == 0
    assert abs(out["eigval"][0, 0]) <= 1e-8 * out["eigval"][0, 1]


def test_65536_generated_trusses():
    torch = _torch()
    from python_stable_3d_truss_analysis_b200 import generate as G
    B = 65536
    gen = G.GenerateRandomCubeTrussesOnDevice(B, seed=31, gridRange=(5, 5, 5), numCubeRange=(7, 7),
                                              isDoStructuralAnalysis=False, asNumpy=False)
    k = 6
    d = {key: gen[key] for key in ("joint_off", "member_off", "xyz", "support", "conn", "aed")}
    fwd = _lib.modes_ragged_device(3, d, k)
    g = torch.ones(B, k, dtype=torch.float64, device="cuda")
    SJ, SM = int(d["support"].numel()), int(d["conn"].numel()) // 2
    res = {"joint_xyz": torch.empty(SJ * 3, dtype=torch.float64, device="cuda"),
           "member_aed": torch.empty(SM * 3, dtype=torch.float64, device="cuda")}
    _lib.modes_adjoint_ragged_device(3, d, fwd, g, res)
    info = fwd["info"].cpu().numpy()
    gen_ok = gen["gen_info"].cpu().numpy() == 0
    assert np.all(info[gen_ok] == 0)
    h = {key: v.cpu().numpy() for key, v in d.items()}
    ev, md, gx, ga = (fwd["eigval"].cpu().numpy(), fwd["modes"].cpu().numpy(), res["joint_xyz"].cpu().numpy(),
                      res["member_aed"].cpu().numpy())
    for b in np.random.default_rng(0).choice(np.nonzero(gen_ok)[0], 24, replace=False):
        j0, j1, m0, m1 = (int(h["joint_off"][b]), int(h["joint_off"][b + 1]), int(h["member_off"][b]),
                          int(h["member_off"][b + 1]))
        joints, support = h["xyz"][3 * j0:3 * j1].reshape(-1, 3), h["support"][j0:j1]
        conn, aed = h["conn"][2 * m0:2 * m1].reshape(-1, 2), h["aed"][3 * m0:3 * m1].reshape(-1, 3)
        vec = md[k * 3 * j0:k * 3 * j1].reshape(k, -1)
        lam_all = modal.modes(3, joints, support, conn, aed)["eigval_all"]
        q = uncut(lam_all, k)
        if q == k:
            check_against_oracle(3, joints, support, conn, aed, ev[b], vec, False, None)
        # the gradient identities of DESIGN section 11: homogeneity in (a, rho) at fixed e, translation invariance
        gab = ga[3 * m0:3 * m1].reshape(-1, 3)
        gxb = gx[3 * j0:3 * j1].reshape(-1, 3)
        lam_sum = ev[b].sum()
        assert abs((gab[:, 1] * aed[:, 1]).sum() - lam_sum) <= 1e-9 * abs(lam_sum)            # lambda is linear in e
        assert np.abs(gxb.sum(0)).max() <= 1e-9 * np.abs(gxb).max() * len(gxb)
        assert abs((gab[:, 0] * aed[:, 0] + gab[:, 2] * aed[:, 2]).sum() + lam_sum) <= 1e-9 * abs(lam_sum) * 4


def test_gradcheck_and_one_launch():
    torch = _torch()
    from python_stable_3d_truss_analysis_b200 import autograd
    ts = [fixture(n)[1:] for n in ("bar-6", "bar-25")]
    p = device(pack(ts))
    base = {key: p[key] for key in ("joint_off", "member_off", "support", "conn")}
    k = int(run(3, pack(ts), 1)["n_free"].max())              # every mode: no cluster is cut
    lam0 = autograd.modes_ragged(base, p["xyz"], p["aed"], n_modes=k)["eigval"]
    w = torch.where(lam0 > 0, 1.0 / lam0.clamp(min=1e-300), torch.zeros_like(lam0))
    SJ = int(p["support"].numel())
    jm0 = torch.full((SJ,), 0.05, dtype=torch.float64, device="cuda")

    def f(dx, sa, sm):                                       # relative sizing and mass, absolute joint shifts
        return (autograd.modes_ragged(base, p["xyz"] + dx, p["aed"] * (1 + sa), jm0 * (1 + sm), n_modes=k)["eigval"] * w).sum()

    z = lambda n: torch.zeros(n, dtype=torch.float64, device="cuda", requires_grad=True)  # noqa: E731
    assert torch.autograd.gradcheck(f, (z(SJ * 3), z(int(p["aed"].numel())), z(SJ)), eps=1e-6, atol=1e-6, rtol=1e-4)
    n0 = _lib.launch_count()
    autograd.modes_ragged(p, n_modes=3, max_joint=64, max_member=200, max_free=60)    # (the packed xyz and aed)
    torch.cuda.synchronize()
    assert _lib.launch_count() - n0 == 1
    with pytest.raises(ValueError):
        autograd.modes_ragged(p, n_modes=0)


def test_cuda_graph_and_consistent_scratch():
    torch = _torch()
    ts = [fixture(n)[1:] for n in ("bar-25", "bar-72")]
    d = device(pack(ts))
    k = 4
    g = torch.ones(2, k, dtype=torch.float64, device="cuda")
    kw = dict(max_joint=int(np.diff(d["joint_off"].cpu().numpy()).max()), max_member=int(np.diff(d["member_off"].cpu().numpy()).max()),
              max_free=150)
    SJ, SM = int(d["support"].numel()), int(d["conn"].numel()) // 2
    fwd = {"eigval": torch.empty(2, k, dtype=torch.float64, device="cuda"), "modes": torch.empty(k * 3 * SJ, dtype=torch.float64, device="cuda"),
           "n_free": torch.empty(2, dtype=torch.int32, device="cuda"), "info": torch.empty(2, dtype=torch.int32, device="cuda")}
    res = {"member_aed": torch.empty(SM * 3, dtype=torch.float64, device="cuda")}
    want = None
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        _lib.modes_ragged_device(3, d, k, out=fwd, **kw)
        _lib.modes_adjoint_ragged_device(3, d, fwd, g, res, **kw)
        want = (fwd["eigval"].clone(), res["member_aed"].clone())
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            _lib.modes_ragged_device(3, d, k, out=fwd, **kw)
            _lib.modes_adjoint_ragged_device(3, d, fwd, g, res, **kw)
    fwd["eigval"].zero_(); res["member_aed"].zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(fwd["eigval"], want[0]) and torch.equal(res["member_aed"], want[1])
    # consistent mass, in a fresh process (the arena is the device's and other calls may have grown it): a capture that
    # would have to grow the arena is refused with nothing enqueued; after a warm-up call the same capture works
    code = """
import numpy as np, torch
from python_stable_3d_truss_analysis_b200 import _lib
from tests.test_gpu_modes_ragged import fixture, pack, device
d = device(pack([fixture(n)[1:] for n in ("bar-25", "bar-72")]))
kw = dict(max_joint=60, max_member=300, max_free=150)
out = {"eigval": torch.full((2, 4), 7.0, dtype=torch.float64, device="cuda"), "modes": None,
       "n_free": torch.empty(2, dtype=torch.int32, device="cuda"), "info": torch.full((2,), 7, dtype=torch.int32, device="cuda")}
s = torch.cuda.Stream()
g = torch.cuda.CUDAGraph()
with torch.cuda.graph(g, stream=s):
    try:
        _lib.modes_ragged_device(3, d, 4, consistent=True, out=out, stream=s, **kw)
        code = 0
    except _lib.TrussLibError as e:
        code = e.code
    out["eigval"].add_(0.0)
g.replay()
torch.cuda.synchronize()
assert code == _lib.TB_ERR_ALLOC and bool((out["eigval"] == 7.0).all()) and bool((out["info"] == 7).all())
with torch.cuda.stream(s):
    _lib.modes_ragged_device(3, d, 4, consistent=True, out=out, stream=s, **kw)
s.synchronize()
want = out["eigval"].clone()
assert bool((out["info"] == 0).all())
out["eigval"].zero_()
g = torch.cuda.CUDAGraph()
with torch.cuda.graph(g, stream=s):
    _lib.modes_ragged_device(3, d, 4, consistent=True, out=out, stream=s, **kw)
g.replay()
torch.cuda.synchronize()
assert torch.equal(out["eigval"], want)
print("graph ok")
"""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, "-c", code], cwd=root, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "graph ok" in res.stdout, res.stdout + res.stderr


def test_host_entry_batch_api_and_dataset(tmp_path):
    from python_stable_3d_truss_analysis_b200.batch import SolveModesBatch
    from python_stable_3d_truss_analysis_b200.dataset import PackedDataset
    from python_stable_3d_truss_analysis_b200.truss import Truss
    ns = ("bar-6", "bar-25", "bar-72")
    ts = [fixture(n)[1:] for n in ns]
    p = pack(ts)
    host = _lib.modes_ragged_host(3, p["joint_off"], p["member_off"], p["xyz"], p["support"], p["conn"], p["aed"], 5,
                                  consistent=True)
    dev = run(3, p, 5, True, max_free=int(host["n_free"].max()))
    for key in ("eigval", "modes", "n_free", "info"):
        assert np.array_equal(host[key], dev[key])
    trusses = [Truss(3).LoadFromJSON(data=json.load(open(f"{H.GOLDEN}/ref_data/{n}_input_0.json"))) for n in ns]
    SolveModesBatch(trusses, nMode=None)
    for b, t in enumerate(trusses):
        one = Truss(3).LoadFromJSON(data=json.load(open(f"{H.GOLDEN}/ref_data/{ns[b]}_input_0.json")))
        one.SolveModes()
        assert np.array_equal(t.GetEigenvalues(), one.GetEigenvalues())
        assert len(t.GetModeShapes()) == len(one.GetModeShapes())
    with pytest.raises(ValueError):
        SolveModesBatch(trusses, nMode=40)                      # bar-6 has fewer free DOFs
    ds = PackedDataset.from_trusses(trusses)
    info = ds.solve_modes(4)
    assert np.all(info == 0)
    path = ds.save(str(tmp_path / "modes.npz"))
    back = PackedDataset.load(path)
    for key in ("eigval", "modes", "n_free", "modes_info"):
        assert np.array_equal(back.a[key], ds.a[key])
    assert np.array_equal(back.truss(1).GetEigenvalues(), ds.a["eigval"][1])
