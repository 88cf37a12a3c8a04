"""Reverse mode of the modal analysis on the GPU (tb_modes_adjoint, k_modes_sens<DIM>, autograd.modes): the kernel's
arithmetic against the numpy eigenvalue gradients fed the device's own eigenpairs on every fixture up to 160 free DOFs,
autograd.modes against central differences of the device forward (simple modes and a loss symmetric in a repeated
pair), gradcheck, the exact identities, bit invariance, failed systems among good ones, CUDA graph capture, the kernel
that ran, and one step of frequency-constrained sizing."""
import numpy as np
import pytest

from oracle import modal
from oracle import modal_adjoint
from oracle import truss_oracle as orc
from python_stable_3d_truss_analysis_b200 import _lib
from tests import helpers as H
from tests import test_modes_adjoint_cpu as CPU
from tests.test_gpu_modes import arrays, fixtures, joint_masses, perturbed, uncut

pytestmark = pytest.mark.gpu

TOL_ARITH = 1e-12    # device vs eigval_grad on the same eigenpairs: the same formulas, other rounding order
TOL_FD = 1e-6
TOL_ID = 1e-11


def _torch():
    import torch
    return torch


def td(a, dt=None):
    torch = _torch()
    return torch.from_numpy(np.ascontiguousarray(a)).to(torch.device("cuda:0"), dt or torch.float64)


def forward(plan, B, xyz, aed, k, consistent=False, jm=None):
    torch = _torch()
    out = {"modes": torch.empty(B, k, plan.N, dtype=torch.float64, device="cuda:0")}
    plan.modes_device(B, xyz, aed=aed, n_modes=k, consistent=consistent, joint_mass=jm, out=out)
    return out


def adjoint(plan, B, xyz, aed, fwd, g, consistent=False):
    torch = _torch()
    f64 = dict(dtype=torch.float64, device="cuda:0")
    res = {"joint_xyz": torch.empty(B, plan.nJ, plan.dim, **f64), "member_aed": torch.empty(B, plan.M, 3, **f64),
           "joint_mass": torch.empty(B, plan.nJ, **f64)}
    plan.modes_adjoint_device(B, xyz, aed, fwd, g, res, consistent=consistent)
    return res


def np_of(d):
    _torch().cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in d.items()}


def grads_of(res, b):
    return res["joint_xyz"][b], res["member_aed"][b], res["joint_mass"][b]


@pytest.mark.parametrize("consistent", [False, True], ids=["lumped", "consistent"])
@pytest.mark.parametrize("name", [f[0] for f in fixtures()])
def test_kernel_against_eigval_grad(name, consistent):
    dim, joints, support, conn, aed = arrays(name)
    plan = _lib.Plan(dim, conn, support)
    rng = np.random.default_rng(17)
    for jm in (None, joint_masses(dim, joints, conn, aed)):
        fwd = forward(plan, 1, td(joints), td(aed), plan.n, consistent, None if jm is None else td(jm))
        g = td(rng.standard_normal((1, plan.n)))
        res = np_of(adjoint(plan, 1, td(joints), td(aed), fwd, g, consistent))
        f = np_of(fwd)
        assert f["info"][0] == 0
        want = modal_adjoint.eigval_grad(dim, joints, support, conn, aed, f["eigval"][0], f["modes"][0], g.cpu().numpy()[0],
                                 consistent)
        CPU.assert_fields_close(grads_of(res, 0), want, TOL_ARITH, name)
        pos = td(rng.uniform(0.5, 1.5, (1, plan.n)))     # identities with a positive cotangent (no cancellation in L)
        res = np_of(adjoint(plan, 1, td(joints), td(aed), fwd, pos, consistent))
        L = float(pos.cpu().numpy()[0] @ f["eigval"][0])
        assert CPU.identities(dim, joints, support, conn, aed, jm, L, grads_of(res, 0)).max() <= TOL_ID


def device_fd(plan, dim, joints, conn, aed, jm, loss, k, consistent, rel):
    """Five-point central differences of loss(eigval[:, :k]) through the device forward: every perturbed system in one
    batch.  Steps as tests/test_modes_adjoint_cpu.fd_gradient."""
    x0 = np.concatenate([joints.ravel(), aed.ravel(), jm])
    nx, na = joints.size, aed.size
    zero = np.empty_like(x0)
    zero[:nx] = np.ptp(joints, axis=0).max()
    zero[nx:nx + na] = 1.0
    zero[nx + na:] = float(np.mean(modal.member_masses(dim, joints, conn, aed)))
    h = rel * np.where(x0 != 0.0, x0, zero)
    P = x0.size
    X = np.tile(x0, (4 * P, 1))
    for s, mult in enumerate((1.0, -1.0, 2.0, -2.0)):
        X[s * P + np.arange(P), np.arange(P)] += mult * h
    fwd = forward(plan, 4 * P, td(X[:, :nx]), td(X[:, nx:nx + na]), k, consistent, td(X[:, nx + na:]))
    f = np_of(fwd)
    assert np.all(f["info"] == 0)
    v = loss(f["eigval"])
    fp, fm, f2p, f2m = v[:P], v[P:2 * P], v[2 * P:3 * P], v[3 * P:]
    d = (8.0 * (fp - fm) - (f2p - f2m)) / (12.0 * h)
    return d[:nx].reshape(joints.shape), d[nx:nx + na].reshape(aed.shape), d[nx + na:]


@pytest.mark.parametrize("name", ["bar-10_input_0", "bar-25_input_0", "bar-72_input_0"])
def test_autograd_simple_modes_against_device_fd(name):
    torch = _torch()
    from python_stable_3d_truss_analysis_b200 import autograd
    from python_stable_3d_truss_analysis_b200.truss import Truss

    dim, joints, support, conn, aed = arrays(name)
    t = Truss(dim).LoadFromJSON(data=H.load_json(f"ref_data/{name}.json"))
    plan = t._get_plan(*t._pack()[1:3])
    jm = joint_masses(dim, joints, conn, aed)
    k = 6
    g = np.random.default_rng(3).standard_normal(k)
    x, a, m = (td(v).requires_grad_(True) for v in (joints, aed, jm))
    out = autograd.modes(t, xyz=x, aed=a, joint_mass=m, n_modes=k)
    (out["eigval"] * td(g)).sum().backward()
    want = device_fd(plan, dim, joints, conn, aed, jm, lambda ev: ev @ g, k, False, CPU.FD_CASES[name])
    CPU.assert_fields_close((x.grad.cpu().numpy(), a.grad.cpu().numpy(), m.grad.cpu().numpy()), want, TOL_FD, name)
    assert not out["modes"].requires_grad and out["info"].dtype == torch.int32


@pytest.mark.parametrize("name", ["bar-72_input_0", "bar-120_input_0"])
def test_autograd_symmetric_penalty_on_a_repeated_pair(name):
    """Sum over modes of relu(lam_min - lambda)^2: equal cotangents on the exactly repeated lowest pair, so the gradient
    is exact whatever basis the forward chose."""
    torch = _torch()
    from python_stable_3d_truss_analysis_b200 import autograd
    from python_stable_3d_truss_analysis_b200.truss import Truss

    dim, joints, support, conn, aed = arrays(name)
    t = Truss(dim).LoadFromJSON(data=H.load_json(f"ref_data/{name}.json"))
    plan = t._get_plan(*t._pack()[1:3])
    lam_all = modal.modes(dim, joints, support, conn, aed)["eigval_all"]
    assert lam_all[1] - lam_all[0] <= 1e-9 * lam_all[0], "the lowest eigenvalue is a pair"
    groups = modal.clusters(lam_all, 1e-9)
    lam_min = 0.5 * (lam_all[groups[1][-1]] + lam_all[groups[2][0]])   # the penalty's kink in a gap of the spectrum
    assert np.abs(lam_all / lam_min - 1.0).min() > 1e-3
    k = uncut(lam_all, 6)
    x, a, m = (td(v).requires_grad_(True) for v in (joints, aed, np.zeros(len(joints))))   # (the gradient at mu = 0)
    out = autograd.modes(t, xyz=x, aed=a, joint_mass=m, n_modes=k)
    torch.relu(lam_min - out["eigval"]).pow(2).sum().backward()

    def pen(ev):
        return (np.maximum(lam_min - ev, 0.0) ** 2).sum(axis=1)

    want = device_fd(plan, dim, joints, conn, aed, np.zeros(len(joints)), pen, k, False, 1e-5)
    CPU.assert_fields_close((x.grad.cpu().numpy(), a.grad.cpu().numpy(), m.grad.cpu().numpy()), want, TOL_FD, name)


def test_autograd_gradcheck():
    torch = _torch()
    from python_stable_3d_truss_analysis_b200 import autograd
    from python_stable_3d_truss_analysis_b200.truss import Truss

    name = "bar-10_input_0"
    dim, joints, support, conn, aed = arrays(name)
    t = Truss(dim).LoadFromJSON(data=H.load_json(f"ref_data/{name}.json"))
    jm = joint_masses(dim, joints, conn, aed) + 0.1 * float(np.mean(modal.member_masses(dim, joints, conn, aed)))
    x0, a0, m0 = td(joints), td(aed), td(jm)
    ref = autograd.modes(t, xyz=x0, aed=a0, joint_mass=m0, n_modes=5)["eigval"]
    span = float(np.ptp(joints, axis=0).max())

    def fn(dx, sa, sm):                          # relative perturbations of every input; outputs O(1)
        return autograd.modes(t, xyz=x0 + span * dx, aed=a0 * sa, joint_mass=m0 * sm, n_modes=5)["eigval"] / ref

    args = (torch.zeros_like(x0, requires_grad=True), torch.ones_like(a0, requires_grad=True),
            torch.ones_like(m0, requires_grad=True))
    assert torch.autograd.gradcheck(fn, args, eps=1e-6, atol=1e-5, rtol=1e-3)


def test_bits_do_not_depend_on_the_launch():
    torch = _torch()
    dim, joints, support, conn, aed = arrays("bar-72_input_0")
    plan = _lib.Plan(dim, conn, support)
    jm = joint_masses(dim, joints, conn, aed)
    B = 5000                                              # more warps than resident ones: the grid-stride loop runs
    A = perturbed(aed, B, 1)
    X = np.tile(joints, (B, 1, 1)) + np.random.default_rng(2).normal(0.0, 0.5, (B,) + joints.shape)
    G = np.random.default_rng(4).standard_normal((B, 6))
    for consistent in (False, True):
        fwd = forward(plan, B, td(X), td(A), 6, consistent, td(jm))
        big = np_of(adjoint(plan, B, td(X), td(A), fwd, td(G), consistent))
        for b in (0, 1, 777, B - 1):
            f1 = forward(plan, 1, td(X[b]), td(A[b]), 6, consistent, td(jm))
            solo = np_of(adjoint(plan, 1, td(X[b]), td(A[b]), f1, td(G[b:b + 1]), consistent))
            for key in solo:
                assert np.array_equal(solo[key][0], big[key][b]), (consistent, b, key)
        sub = {k: v[700:1000].contiguous() for k, v in fwd.items()}
        mid = np_of(adjoint(plan, 300, td(X[700:1000]), td(A[700:1000]), sub, td(G[700:1000]), consistent))
        for key in mid:
            assert np.array_equal(mid[key], big[key][700:1000]), key
        # stride-0 shared inputs == the same rows repeated
        fs = forward(plan, 40, td(X[5]), td(A[5]), 6, consistent, td(jm))
        sh = np_of(adjoint(plan, 40, td(X[5]), td(A[5]), fs, td(np.tile(G[5], (40, 1))), consistent))
        fr = forward(plan, 40, td(np.tile(X[5], (40, 1, 1))), td(np.tile(A[5], (40, 1, 1))), 6, consistent,
                     td(np.tile(jm, (40, 1))))
        rep = np_of(adjoint(plan, 40, td(np.tile(X[5], (40, 1, 1))), td(np.tile(A[5], (40, 1, 1))), fr,
                            td(np.tile(G[5], (40, 1))), consistent))
        for key in sh:
            assert np.array_equal(sh[key], rep[key]) and np.array_equal(sh[key][3], big[key][5]), key
        # n_modes = 6 with g == n_modes = n with g padded by zeros (modes with g = 0 are skipped)
        fa = forward(plan, 64, td(X[:64]), td(A[:64]), plan.n, consistent, td(jm))
        Gp = np.zeros((64, plan.n))
        Gp[:, :6] = G[:64]
        full = np_of(adjoint(plan, 64, td(X[:64]), td(A[:64]), fa, td(Gp), consistent))
        for key in full:
            assert np.array_equal(full[key], big[key][:64]), key
    torch.cuda.synchronize()


@pytest.mark.parametrize("consistent", [False, True], ids=["lumped", "consistent"])
def test_failed_systems_get_zero_gradients(consistent):
    dim, joints, support, conn, aed = arrays("bar-72_input_0")
    plan = _lib.Plan(dim, conn, support)
    B = 3000
    A = perturbed(aed, B, 7)
    X = np.tile(joints, (B, 1, 1))
    want = {11: -2}
    X[11, conn[4, 1]] = X[11, conn[4, 0]]                      # zero-length member
    free_joint = int(np.nonzero(support == orc.NO)[0][0])
    for b in (12, 1500, 2999):                                 # no mass at a free joint
        A[b, (conn == free_joint).any(axis=1), 2] = 0.0
        want[b] = _lib.TB_INFO_MASS
    G = np.random.default_rng(8).standard_normal((B, 8))
    fwd = forward(plan, B, td(X), td(A), 8, consistent)
    res = adjoint(plan, B, td(X), td(A), fwd, td(G), consistent)
    res = np_of(res)
    info = fwd["info"].cpu().numpy()
    for b in range(B):
        assert info[b] == want.get(b, 0), b
    for b in want:
        for key in res:
            assert not res[key][b].any() and np.all(np.isfinite(res[key][b])), (b, key)
    for b in (10, 13, 1499, 2998):
        f1 = forward(plan, 1, td(X[b]), td(A[b]), 8, consistent)
        solo = np_of(adjoint(plan, 1, td(X[b]), td(A[b]), f1, td(G[b:b + 1]), consistent))
        for key in solo:
            assert np.array_equal(solo[key][0], res[key][b]), (b, key)


def test_forward_and_adjoint_in_one_cuda_graph():
    torch = _torch()
    dim, joints, support, conn, aed = arrays("bar-72_input_0")
    A = perturbed(aed, 600, 5)
    xyz, aedt = td(joints), td(A)
    G = td(np.random.default_rng(6).standard_normal((600, 6)))
    s = torch.cuda.Stream()
    for consistent in (False, True):
        plan = _lib.Plan(dim, conn, support)
        f64 = dict(dtype=torch.float64, device="cuda:0")
        fwd = {"eigval": torch.empty(600, 6, **f64), "info": torch.empty(600, dtype=torch.int32, device="cuda:0"),
               "modes": torch.empty(600, 6, plan.N, **f64)}
        res = {"joint_xyz": torch.empty(600, plan.nJ, dim, **f64), "member_aed": torch.empty(600, plan.M, 3, **f64),
               "joint_mass": torch.empty(600, plan.nJ, **f64)}

        def step():
            plan.modes_device(600, xyz, aed=aedt, n_modes=6, consistent=consistent, out=fwd, stream=s)
            plan.modes_adjoint_device(600, xyz, aedt, fwd, G, res, consistent=consistent, stream=s)

        if consistent:                                      # warm-up outside the capture: grows the consistent-mass slots
            with torch.cuda.stream(s):
                step()
        s.synchronize()
        with torch.cuda.stream(s):
            step()
        s.synchronize()
        want = {k: v.clone() for k, v in res.items()}
        for v in list(res.values()) + list(fwd.values()):
            v.zero_()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            step()
        g.replay()
        torch.cuda.synchronize()
        for k in want:
            assert torch.equal(res[k], want[k]), (consistent, k)


def test_profiler_shows_k_modes_sens():
    torch = _torch()
    from torch.profiler import ProfilerActivity, profile

    dim, joints, support, conn, aed = arrays("bar-25_input_0")
    plan = _lib.Plan(dim, conn, support)
    fwd = forward(plan, 16, td(joints), td(perturbed(aed, 16, 2)), 4)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        adjoint(plan, 16, td(joints), td(perturbed(aed, 16, 2)), fwd, td(np.ones((16, 4))))
        torch.cuda.synchronize()
    assert _lib.launch_count() - n0 == 1                    # one native launch
    names = [ev.name for ev in prof.events()]
    assert any("k_modes_sens" in n for n in names), sorted(set(names))


def test_sizing_step_decreases_weight_plus_frequency_penalty():
    """bar-72, areas as design variables: loss = weight + c * sum relu(lam_min - lambda)^2 (lambda from autograd.modes,
    the weight from autograd.solve); one step along -grad decreases it."""
    torch = _torch()
    from python_stable_3d_truss_analysis_b200 import autograd
    from python_stable_3d_truss_analysis_b200.truss import Truss

    t = Truss(3).LoadFromJSON(data=H.load_json("ref_data/bar-72_input_0.json"))
    aed0 = td(t._pack()[3])
    lam0 = autograd.modes(t, aed=aed0, n_modes=8)["eigval"].detach()
    lam_min = float(lam0[2]) * 1.2                           # the lowest modes violate the constraint
    w0 = float(autograd.solve(t, aed=aed0)["weight"])
    c = w0 / float(lam_min) ** 2 * 10.0

    def loss(area):
        aed = torch.cat([area[:, None], aed0[:, 1:]], 1)
        lam = autograd.modes(t, aed=aed, n_modes=8)["eigval"]
        return autograd.solve(t, aed=aed)["weight"] + c * torch.relu(lam_min - lam).pow(2).sum()

    area = aed0[:, 0].clone().requires_grad_(True)
    L0 = loss(area)
    L0.backward()
    g = area.grad
    step = 0.01 * float(area.detach().abs().max()) / float(g.abs().max())
    L1 = loss((area - step * g).detach())
    assert float(L1) < float(L0.detach())


def test_autograd_argument_shapes_and_batch_sizes():
    torch = _torch()
    from python_stable_3d_truss_analysis_b200 import autograd
    from python_stable_3d_truss_analysis_b200.truss import Truss

    t = Truss(3).LoadFromJSON(data=H.load_json("ref_data/bar-72_input_0.json"))
    joints, _, _, aed, _ = t._pack()
    with pytest.raises(ValueError):
        autograd.modes(t, xyz=td(joints[:-1]))
    with pytest.raises(ValueError):
        autograd.modes(t, aed=td(aed[:, :2]))
    with pytest.raises(ValueError):
        autograd.modes(t, joint_mass=td(np.ones(t.nJoint + 1)))
    with pytest.raises(ValueError):                                        # batch sizes disagree
        autograd.modes(t, xyz=td(np.tile(joints, (3, 1, 1))), aed=td(np.tile(aed, (4, 1, 1))))
    with pytest.raises(ValueError):
        autograd.modes(t, aed=td(np.tile(aed, (3, 1, 1))), joint_mass=td(np.ones((2, t.nJoint))))
    with pytest.raises(TypeError):
        autograd.modes(t, xyz=td(joints), aed=td(aed).to(torch.float32))
    out = autograd.modes(t, aed=td(np.tile(aed, (3, 1, 1))), joint_mass=td(np.ones(t.nJoint)), n_modes=4)
    assert tuple(out["eigval"].shape) == (3, 4) and tuple(out["modes"].shape) == (3, 4, 3 * t.nJoint)
    one = autograd.modes(t, n_modes=4)
    assert tuple(one["eigval"].shape) == (4,) and one["info"].dim() == 0
