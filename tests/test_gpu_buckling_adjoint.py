"""Reverse mode of linear buckling on the GPU (tb_buckling_adjoint, k_buckling_sens<DIM>, autograd.buckling): the
kernel's arithmetic against the numpy load-factor gradients fed the device's own factors and modes on every fixture up
to 160 free DOFs, the exact identities (explicit and through tb_adjoint), autograd.buckling against central differences
of the device forward (static solve, then buckling), gradcheck, bit invariance, failed systems among good ones, infinite
factors, one CUDA graph for both forwards and both adjoints, the launches, and one step of stability-constrained sizing."""
import numpy as np
import pytest

from oracle import buckling_adjoint as badj
from oracle import modal
from oracle import truss_oracle as orc
from python_stable_3d_truss_analysis_b200 import _lib
from tests import helpers as H
from tests import test_buckling_adjoint_cpu as CPU
from tests.test_gpu_buckling import perturbed, td

pytestmark = pytest.mark.gpu

TOL_ARITH = 1e-12    # device vs factor_grad on the same factors and modes: the same formulas, other rounding order
TOL_FD = 1e-6
TOL_ID = 1e-11


def _torch():
    import torch
    return torch


def f64():
    torch = _torch()
    return dict(dtype=torch.float64, device="cuda:0")


def forward(plan, B, xyz, aed, force, k):
    """Static solve, then buckling under its member forces: (static outputs, buckling outputs) on the device."""
    torch = _torch()
    st = {"u": torch.empty(B, plan.N, **f64()), "axial": torch.empty(B, plan.M, **f64()),
          "info": torch.empty(B, dtype=torch.int32, device="cuda:0")}
    plan.solve_device(B, xyz, force, aed=aed, out=st)
    bo = {"modes": torch.empty(B, k, plan.N, **f64())}
    plan.buckling_device(B, xyz, st["axial"], aed=aed, n_modes=k, out=bo)
    return st, bo


def adjoint(plan, B, xyz, aed, axial, fwd, g, **kw):
    torch = _torch()
    res = {"joint_xyz": torch.empty(B, plan.nJ, plan.dim, **f64()), "member_aed": torch.empty(B, plan.M, 3, **f64()),
           "axial": torch.empty(B, plan.M, **f64())}
    plan.buckling_adjoint_device(B, xyz, aed, axial, fwd, g, res, **kw)
    return res


def static_adjoint(plan, B, xyz, aed, force, u, g_axial):
    """tb_adjoint with the cotangent g_axial on the member forces: the share of the gradients through N."""
    torch = _torch()
    res = {"joint_xyz": torch.empty(B, plan.nJ, plan.dim, **f64()), "member_aed": torch.empty(B, plan.M, 3, **f64()),
           "force": torch.empty(B, plan.N, **f64())}
    plan.adjoint_device(B, xyz, force, aed, u, {"axial": g_axial}, res)
    return res


def np_of(d):
    _torch().cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in d.items()}


@pytest.mark.parametrize("name", list(CPU.CASES))
def test_kernel_against_factor_grad_and_the_identities(name):
    dim, joints, support, conn, aed, force = CPU.CASES[name]
    plan = _lib.Plan(dim, conn, support)
    st, bo = forward(plan, 1, td(joints), td(aed), td(force), plan.n)
    rng = np.random.default_rng(17)
    g = td(rng.standard_normal((1, plan.n)))
    res = np_of(adjoint(plan, 1, td(joints), td(aed), st["axial"], bo, g))
    f, s = np_of(bo), np_of(st)
    assert s["info"][0] == 0 and f["info"][0] == 0
    ax = s["axial"][0]
    want = badj.factor_grad(dim, joints, support, conn, aed, ax, f["factor"][0], f["modes"][0], g.cpu().numpy()[0])
    for key, w in zip(("joint_xyz", "member_aed", "axial"), want):
        err = orc.normwise_err(res[key][0].ravel(), w.ravel())
        assert err <= TOL_ARITH, (name, key, err)
    assert not res["member_aed"][0][:, 2].any()
    # identities, explicit and through tb_adjoint, with positive cotangents on the clearly critical factors
    gp = CPU.clear_cotangent(CPU.forward(name)[-1], 5)
    L = float(gp @ np.where(gp != 0.0, f["factor"][0], 0.0))
    res = adjoint(plan, 1, td(joints), td(aed), st["axial"], bo, td(gp[None]))
    tot = np_of(static_adjoint(plan, 1, td(joints), td(aed), td(force), st["u"], res["axial"]))
    res = np_of(res)
    explicit = (res["joint_xyz"][0], res["member_aed"][0], res["axial"][0])
    total = (explicit[0] + tot["joint_xyz"][0], explicit[1] + tot["member_aed"][0], tot["force"][0])
    assert CPU.identities(dim, joints, support, conn, aed, force, ax, L, explicit, total).max() <= TOL_ID


def device_fd(plan, dim, joints, aed, force, loss, k):
    """Five-point central differences of loss(factor[:, :k]) through the device forward (static solve, then buckling),
    every perturbed system in one batch; steps as tests/test_buckling_adjoint_cpu.py."""
    nx, na, nf = joints.size, len(aed), force.size
    x0 = np.concatenate([joints.ravel(), aed[:, 0], aed[:, 1], force])
    h = CPU.FD_REL * np.concatenate([np.full(nx, np.ptp(joints, axis=0).max()), aed[:, 0], aed[:, 1],
                                     np.full(nf, np.abs(force).max())])
    P = x0.size
    X = np.tile(x0, (4 * P, 1))
    for s, mult in enumerate((1.0, -1.0, 2.0, -2.0)):
        X[s * P + np.arange(P), np.arange(P)] += mult * h
    A = np.stack([X[:, nx:nx + na], X[:, nx + na:nx + 2 * na], np.tile(aed[:, 2], (4 * P, 1))], 2)
    st, bo = forward(plan, 4 * P, td(X[:, :nx].reshape(4 * P, -1, dim)), td(A), td(X[:, nx + 2 * na:]), k)
    f = np_of(bo)
    assert np.all(f["info"] == 0)
    v = loss(f["factor"])
    fp, fm, f2p, f2m = v[:P], v[P:2 * P], v[2 * P:3 * P], v[3 * P:]
    d = (8.0 * (fp - fm) - (f2p - f2m)) / (12.0 * h)
    return d[:nx].reshape(joints.shape), np.stack([d[nx:nx + na], d[nx + na:nx + 2 * na]], 1), d[nx + 2 * na:]


@pytest.mark.parametrize("name", ["bar-10_input_0", "bar-25_input_0", "bar-47_input_0", "bar-72_input_0"])
def test_autograd_against_device_fd(name):
    """loss = the sum of the lowest cluster of factors (one factor, or bar-72_input_0's exactly repeated pair: a
    symmetric cotangent), differentiated through the static solve to the joints, the members and the loads."""
    torch = _torch()
    from python_stable_3d_truss_analysis_b200 import autograd
    from python_stable_3d_truss_analysis_b200.truss import Truss

    dim, joints, support, conn, aed, force = CPU.CASES[name]
    t = Truss(dim).LoadFromJSON(data=H.load_json(f"ref_data/{name}.json"))
    plan = t._get_plan(*t._pack()[1:3])
    r = CPU.forward(name)[-1]
    fac = r["factor_all"]
    low = modal.clusters(fac[np.isfinite(fac)], 1e-6)[0]
    k = low[-1] + 2
    x, a, fo = (td(v).requires_grad_(True) for v in (joints, aed, force))
    out = autograd.buckling(t, xyz=x, aed=a, force=fo, n_modes=k)
    out["factor"][low].sum().backward()
    want = device_fd(plan, dim, joints, aed, force, lambda fac: fac[:, low].sum(axis=1), k)
    mask = orc.free_mask(dim, support)
    CPU.assert_close(x.grad.cpu().numpy(), want[0], TOL_FD, f"{name} xyz")
    CPU.assert_close(a.grad.cpu().numpy()[:, :2], want[1], TOL_FD, f"{name} (a, E)")
    CPU.assert_close(fo.grad.cpu().numpy()[mask], want[2][mask], TOL_FD, f"{name} force")
    assert not a.grad[:, 2].any() and not fo.grad.cpu().numpy()[~mask].any()
    assert not out["modes"].requires_grad and out["info"].dtype == torch.int32 and out["axial"].requires_grad


def test_autograd_gradcheck():
    torch = _torch()
    from python_stable_3d_truss_analysis_b200 import autograd
    from python_stable_3d_truss_analysis_b200.truss import Truss

    name = "bar-10_input_0"
    dim, joints, support, conn, aed, force = CPU.CASES[name]
    t = Truss(dim).LoadFromJSON(data=H.load_json(f"ref_data/{name}.json"))
    x0, a0, f0 = td(joints), td(aed), td(force)
    ref = autograd.buckling(t, xyz=x0, aed=a0, force=f0, n_modes=3)["factor"]
    assert bool(torch.isfinite(ref).all())
    span = float(np.ptp(joints, axis=0).max())

    def fn(dx, sa, sf):                          # relative perturbations of every input; outputs O(1)
        return autograd.buckling(t, xyz=x0 + span * dx, aed=a0 * sa, force=f0 * sf, n_modes=3)["factor"] / ref

    args = (torch.zeros_like(x0, requires_grad=True), torch.ones_like(a0, requires_grad=True),
            torch.ones_like(f0, requires_grad=True))
    assert torch.autograd.gradcheck(fn, args, eps=1e-6, atol=1e-5, rtol=1e-3)
    ax = autograd.buckling(t, xyz=x0, aed=a0, force=f0)["axial"].detach()   # given member forces: N is an input
    assert torch.autograd.gradcheck(lambda s: autograd.buckling(t, xyz=x0, aed=a0, axial=ax * s, n_modes=3)["factor"] / ref,
                                    (torch.ones_like(ax, requires_grad=True),), eps=1e-6, atol=1e-5, rtol=1e-3)


def test_bits_do_not_depend_on_the_launch():
    torch = _torch()
    dim, joints, support, conn, aed, force = CPU.CASES["bar-72_input_0"]
    plan = _lib.Plan(dim, conn, support)
    B = 5000                                              # more warps than resident ones: the grid-stride loop runs
    A = perturbed(aed, B, 1)
    X = np.tile(joints, (B, 1, 1)) + np.random.default_rng(2).normal(0.0, 0.5, (B,) + joints.shape)
    G = np.random.default_rng(4).standard_normal((B, 6))
    st, bo = forward(plan, B, td(X), td(A), td(force), 6)
    AX = st["axial"]
    assert not st["info"].any() and not bo["info"].any()
    big = np_of(adjoint(plan, B, td(X), td(A), AX, bo, td(G)))
    for b in (0, 1, 777, B - 1):
        sub = {k: v[b:b + 1].contiguous() for k, v in bo.items()}
        solo = np_of(adjoint(plan, 1, td(X[b]), td(A[b]), AX[b:b + 1].contiguous(), sub, td(G[b:b + 1])))
        for key in solo:
            assert np.array_equal(solo[key][0], big[key][b]), (b, key)
    sub = {k: v[700:1000].contiguous() for k, v in bo.items()}
    mid = np_of(adjoint(plan, 300, td(X[700:1000]), td(A[700:1000]), AX[700:1000].contiguous(), sub, td(G[700:1000])))
    for key in mid:
        assert np.array_equal(mid[key], big[key][700:1000]), key
    # stride-0 shared inputs (the member forces included) == the same rows repeated
    ax5 = AX[5].contiguous()
    fs = {"modes": torch.empty(40, 6, plan.N, **f64())}
    plan.buckling_device(40, td(X[5]), ax5, aed=td(A[5]), n_modes=6, out=fs)
    sh = np_of(adjoint(plan, 40, td(X[5]), td(A[5]), ax5, fs, td(np.tile(G[5], (40, 1)))))
    rep_ax = ax5.repeat(40, 1)
    fr = {"modes": torch.empty(40, 6, plan.N, **f64())}
    plan.buckling_device(40, td(np.tile(X[5], (40, 1, 1))), rep_ax, aed=td(np.tile(A[5], (40, 1, 1))), n_modes=6, out=fr)
    rep = np_of(adjoint(plan, 40, td(np.tile(X[5], (40, 1, 1))), td(np.tile(A[5], (40, 1, 1))), rep_ax, fr,
                        td(np.tile(G[5], (40, 1)))))
    for key in sh:
        assert np.array_equal(sh[key], rep[key]) and np.array_equal(sh[key][3], big[key][5]), key
    # an explicit axial stride: every other row of a [2B, M] array
    wide = torch.zeros(80, plan.M, **f64())
    wide[::2] = AX[:40]
    sub = {k: v[:40].contiguous() for k, v in bo.items()}
    sd = np_of(adjoint(plan, 40, td(X[:40]), td(A[:40]), wide, sub, td(G[:40]), axial_stride=2 * plan.M))
    for key in sd:
        assert np.array_equal(sd[key], big[key][:40]), key
    # n_modes = 6 == n_modes = n with the cotangent padded by zeros (modes with g = 0 are skipped)
    fa = {"modes": torch.empty(64, plan.n, plan.N, **f64())}
    plan.buckling_device(64, td(X[:64]), AX[:64].contiguous(), aed=td(A[:64]), out=fa)
    Gp = np.zeros((64, plan.n))
    Gp[:, :6] = G[:64]
    full = np_of(adjoint(plan, 64, td(X[:64]), td(A[:64]), AX[:64].contiguous(), fa, td(Gp)))
    for key in full:
        assert np.array_equal(full[key], big[key][:64]), key


def test_failed_systems_and_infinite_factors_get_zero_gradients():
    torch = _torch()
    dim, joints, support, conn, aed, force = CPU.CASES["bar-72_input_0"]
    plan = _lib.Plan(dim, conn, support)
    B = 3000
    A = perturbed(aed, B, 7)
    X = np.tile(joints, (B, 1, 1))
    X[11, conn[4, 1]] = X[11, conn[4, 0]]                     # zero-length member
    free_joint = int(np.nonzero(support == orc.NO)[0][0])
    mech = (12, 1500, 2999)
    for b in mech:                                            # no stiffness at a free joint: a mechanism
        A[b, (conn == free_joint).any(axis=1), 1] = 0.0
    st, _ = forward(plan, B, td(X), td(A), td(force), 8)
    AX = st["axial"].clone()
    AX[20] = 0.0                                              # zero forces: every factor +inf, info 0
    AX[22] = 0.0
    bo = {"modes": torch.empty(B, 8, plan.N, **f64())}
    plan.buckling_device(B, td(X), AX, aed=td(A), n_modes=8, out=bo)
    info = bo["info"].cpu().numpy()
    assert info[11] == -2 and all(info[b] > 0 for b in mech) and np.count_nonzero(info) == 1 + len(mech)
    fac = bo["factor"].cpu().numpy()
    assert np.all(np.isinf(fac[20])) and np.all(np.isinf(fac[22]))
    G = np.random.default_rng(8).standard_normal((B, 8))     # (a nonzero cotangent on system 22's infinite factors)
    G[20] = np.inf                                            # an infinite cotangent on infinite factors
    res = np_of(adjoint(plan, B, td(X), td(A), AX, bo, td(G)))
    for b in (11, 20, 22) + mech:
        for key in res:
            assert not res[key][b].any(), (b, key)
    for key in res:
        assert np.all(np.isfinite(res[key])), key
    for b in (10, 13, 21, 1499, 2998):                         # good neighbours == the system alone
        sub = {k: v[b:b + 1].contiguous() for k, v in bo.items()}
        solo = np_of(adjoint(plan, 1, td(X[b]), td(A[b]), AX[b:b + 1].contiguous(), sub, td(G[b:b + 1])))
        for key in solo:
            assert np.array_equal(solo[key][0], res[key][b]), (b, key)
    # the counting rule: a 2D triangle with one pin and nothing else
    j = np.array([[0.0, 0.0], [4.0, 0.0], [2.0, 3.0]])
    tri = _lib.Plan(2, np.array([[0, 1], [1, 2], [0, 2]], np.int32), np.array([orc.PIN, 0, 0], np.uint8))
    a3, n3 = td(np.tile([1.0, 1e7, 0.1], (3, 1))), td(np.full(3, -1.0))
    fo = {"modes": torch.empty(5, 2, tri.N, **f64())}
    tri.buckling_device(5, td(j), n3, aed=a3, n_modes=2, out=fo)
    assert bool((fo["info"] == -1).all())
    rt = {"joint_xyz": torch.full((5, 3, 2), 7.0, **f64()), "member_aed": torch.full((5, 3, 3), 7.0, **f64()),
          "axial": torch.full((5, 3), 7.0, **f64())}
    tri.buckling_adjoint_device(5, td(j), a3, n3, fo, td(np.ones((5, 2))), rt)
    for key, v in np_of(rt).items():
        assert not v.any(), key


def test_both_forwards_and_both_adjoints_in_one_cuda_graph():
    torch = _torch()
    dim, joints, support, conn, aed, force = CPU.CASES["bar-72_input_0"]
    plan = _lib.Plan(dim, conn, support)
    B = 600
    xyz, aedt, ft = td(joints), td(perturbed(aed, B, 5)), td(force)
    G = td(np.random.default_rng(6).standard_normal((B, 6)))
    st = {"u": torch.empty(B, plan.N, **f64()), "axial": torch.empty(B, plan.M, **f64()),
          "info": torch.empty(B, dtype=torch.int32, device="cuda:0")}
    bo = {"factor": torch.empty(B, 6, **f64()), "modes": torch.empty(B, 6, plan.N, **f64()),
          "info": torch.empty(B, dtype=torch.int32, device="cuda:0")}
    bres = {"joint_xyz": torch.empty(B, plan.nJ, dim, **f64()), "member_aed": torch.empty(B, plan.M, 3, **f64()),
            "axial": torch.empty(B, plan.M, **f64())}
    sres = {"joint_xyz": torch.empty(B, plan.nJ, dim, **f64()), "member_aed": torch.empty(B, plan.M, 3, **f64()),
            "force": torch.empty(B, plan.N, **f64())}
    s = torch.cuda.Stream()

    def step():
        plan.solve_device(B, xyz, ft, aed=aedt, out=st, stream=s)
        plan.buckling_device(B, xyz, st["axial"], aed=aedt, n_modes=6, out=bo, stream=s)
        plan.buckling_adjoint_device(B, xyz, aedt, st["axial"], bo, G, bres, stream=s)
        plan.adjoint_device(B, xyz, ft, aedt, st["u"], {"axial": bres["axial"]}, sres, stream=s)

    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):                                # warm-up outside the capture: grows the arenas
        step()
    s.synchronize()
    assert not st["info"].any() and not bo["info"].any()
    want = {(i, k): v.clone() for i, d in enumerate((bres, sres)) for k, v in d.items()}
    for d in (st, bo, bres, sres):
        for v in d.values():
            v.zero_()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        step()
    g.replay()
    torch.cuda.synchronize()
    for (i, k), v in want.items():
        assert torch.equal((bres, sres)[i][k], v), (i, k)


def test_launches_and_the_kernel_that_ran():
    torch = _torch()
    from torch.profiler import ProfilerActivity, profile
    from python_stable_3d_truss_analysis_b200 import autograd
    from python_stable_3d_truss_analysis_b200.truss import Truss

    name = "bar-25_input_0"
    dim, joints, support, conn, aed, force = CPU.CASES[name]
    t = Truss(dim).LoadFromJSON(data=H.load_json(f"ref_data/{name}.json"))
    plan = t._get_plan(*t._pack()[1:3])
    A = td(perturbed(aed, 16, 2))
    st, bo = forward(plan, 16, td(joints), A, td(force), 4)
    g = td(np.ones((16, 4)))
    adjoint(plan, 16, td(joints), A, st["axial"], bo, g)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = adjoint(plan, 16, td(joints), A, st["axial"], bo, g)
        torch.cuda.synchronize()
    assert _lib.launch_count() - n0 == 1                    # one native launch
    names = [ev.name for ev in prof.events()]
    assert any("k_buckling_sens" in n for n in names), sorted(set(names))
    static_adjoint(plan, 16, td(joints), A, td(force), st["u"], res["axial"])
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    static_adjoint(plan, 16, td(joints), A, td(force), st["u"], res["axial"])
    torch.cuda.synchronize()
    n_adj = _lib.launch_count() - n0
    x = td(joints).requires_grad_(True)                      # (every input: the gradients static_adjoint writes)
    a = A.clone().requires_grad_(True)
    f = td(force).requires_grad_(True)
    out = autograd.buckling(t, xyz=x, aed=a, force=f, n_modes=4)
    loss = out["factor"].sum()
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    loss.backward()
    torch.cuda.synchronize()
    assert _lib.launch_count() - n0 == 1 + n_adj             # tb_buckling_adjoint, then tb_adjoint's launches
    assert x.grad is not None and a.grad is not None and f.grad is not None


def test_sizing_step_decreases_weight_plus_buckling_penalty():
    """bar-72, areas as design variables: loss = weight + c * sum relu(target - factor) with the target above the
    lowest (repeated) factor, so the penalty is active and symmetric in the pair; one step along -grad decreases it."""
    torch = _torch()
    from python_stable_3d_truss_analysis_b200 import autograd
    from python_stable_3d_truss_analysis_b200.truss import Truss

    t = Truss(3).LoadFromJSON(data=H.load_json("ref_data/bar-72_input_0.json"))
    aed0 = td(t._pack()[3])
    fac0 = autograd.buckling(t, aed=aed0, n_modes=6)["factor"].detach()
    target = float(fac0[0]) * 1.2
    w0 = float(autograd.solve(t, aed=aed0)["weight"])
    c = w0 / target * 10.0

    def loss(area):
        aed = torch.cat([area[:, None], aed0[:, 1:]], 1)
        fac = autograd.buckling(t, aed=aed, n_modes=6)["factor"]
        return autograd.solve(t, aed=aed)["weight"] + c * torch.relu(target - fac).sum()

    area = aed0[:, 0].clone().requires_grad_(True)
    L0 = loss(area)
    L0.backward()
    g = area.grad
    assert bool(torch.isfinite(g).all()) and float(g.abs().max()) > 0.0
    step = 0.01 * float(area.detach().abs().max()) / float(g.abs().max())
    L1 = loss((area - step * g).detach())
    assert float(L1) < float(L0.detach())


def test_autograd_argument_shapes_and_batch_sizes():
    torch = _torch()
    from python_stable_3d_truss_analysis_b200 import autograd
    from python_stable_3d_truss_analysis_b200.truss import Truss

    t = Truss(3).LoadFromJSON(data=H.load_json("ref_data/bar-72_input_0.json"))
    joints, _, _, aed, force = t._pack()
    with pytest.raises(ValueError):
        autograd.buckling(t, xyz=td(joints[:-1]))
    with pytest.raises(ValueError):
        autograd.buckling(t, aed=td(aed[:, :2]))
    with pytest.raises(ValueError):
        autograd.buckling(t, axial=td(np.ones(t.nMember + 1)))
    with pytest.raises(ValueError):
        autograd.buckling(t, force=td(np.ones(force.size + 1)))
    with pytest.raises(ValueError):                                        # batch sizes disagree
        autograd.buckling(t, xyz=td(np.tile(joints, (3, 1, 1))), aed=td(np.tile(aed, (4, 1, 1))))
    with pytest.raises(ValueError):
        autograd.buckling(t, aed=td(np.tile(aed, (3, 1, 1))), force=td(np.tile(force, (2, 1))))
    out = autograd.buckling(t, aed=td(np.tile(aed, (3, 1, 1))), n_modes=4)
    assert tuple(out["factor"].shape) == (3, 4) and tuple(out["modes"].shape) == (3, 4, 3 * t.nJoint)
    assert tuple(out["axial"].shape) == (3, t.nMember) and tuple(out["info"].shape) == (3,)
    one = autograd.buckling(t, n_modes=4)
    assert tuple(one["factor"].shape) == (4,) and one["info"].dim() == 0 and tuple(one["axial"].shape) == (t.nMember,)
    given = autograd.buckling(t, axial=one["axial"], n_modes=4)             # the same member forces, given
    assert torch.equal(given["factor"], one["factor"])
