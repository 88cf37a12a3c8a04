"""Modal analysis on the GPU (tb_modes / tb_modes_host, k_modes<DIM>): eigenvalues and mode shapes against the numpy
oracle (oracle/modal.py) on every fixture up to 160 free DOFs, both mass models, with and without joint masses; bit
invariance under batch position, batch size, strides, gene tables and n_modes; failures among good systems; the
consistent-mass scratch under CUDA graph capture; and the Python API."""
import numpy as np
import pytest

from oracle import modal
from oracle import truss_oracle as orc
from python_stable_3d_truss_analysis_b200 import _lib
from tests import helpers as H

pytestmark = pytest.mark.gpu

TOL_VAL = 1e-11      # |lambda - lambda_ref| <= TOL_VAL * lambda_max, residual, M-orthonormality
TOL_VEC = 1e-8       # isolated vectors and cluster projectors


def fixtures():
    return [(n, d, data) for n, d, data, _ in H.shipped_cases() if not n.startswith("bar-942")] + \
        [(n, d, data) for n, d, data, _ in H.cube7_shipped()[:2]]


def arrays(name):
    for n, d, data in fixtures():
        if n == name:
            return (d,) + tuple(orc.arrays_from_json(data, d)[:4])
    raise KeyError(name)


def joint_masses(dim, joints, conn, aed):
    return np.linspace(0.0, 3.0, len(joints)) * float(np.mean(modal.member_masses(dim, joints, conn, aed)))


def check_against_oracle(dim, joints, support, conn, aed, got_val, got_vec, consistent, jm):
    """Every check of one system; returns the largest |lambda - lambda_ref| / lambda_ref over the returned modes."""
    ref = modal.modes(dim, joints, support, conn, aed, consistent=consistent, joint_mass=jm)
    K, Mf, mask = ref["K_ff"], ref["M_ff"], ref["mask"]
    lam_all = ref["eigval_all"]
    lmax = np.abs(lam_all).max()
    k = len(got_val)
    assert np.abs(got_val - lam_all[:k]).max() <= TOL_VAL * lmax
    assert np.all(got_vec[:, ~mask] == 0.0)
    phi = got_vec[:, mask].T                               # [n, k]
    Mphi = Mf @ phi
    assert np.abs(K @ phi - Mphi * got_val).max() <= TOL_VAL * lmax * np.abs(Mphi).max()
    assert np.abs(phi.T @ Mphi - np.eye(k)).max() <= TOL_VAL
    big = np.argmax(np.abs(phi), axis=0)
    assert np.all(phi[big, np.arange(k)] > 0)
    ref_phi = ref["modes"][:k][:, mask].T
    for g in modal.clusters(lam_all, 1e-6):
        if g[-1] >= k:                                     # (a cluster cut by n_modes: eigenvalues and residuals only)
            continue
        if len(g) == 1:
            a, b = phi[:, g[0]], ref_phi[:, g[0]]
            mags = np.sort(np.abs(b))[::-1]
            if len(mags) > 1 and mags[0] - mags[1] <= 1e-8 * mags[0]:
                b = b * np.sign(a @ Mf @ b)                 # a near tie of the largest components: the sign is rounding's
            assert np.linalg.norm(a - b) <= TOL_VEC * np.linalg.norm(b)
        else:                                              # a cluster: its M-projector
            P = phi[:, g] @ phi[:, g].T @ Mf
            Pr = ref_phi[:, g] @ ref_phi[:, g].T @ Mf
            assert np.abs(P - Pr).max() <= TOL_VEC * max(1.0, np.abs(Pr).max())
    return float(np.max(np.abs(got_val - lam_all[:k]) / np.abs(lam_all[:k]).clip(1e-300)))


def uncut(lam_all, k):
    """The smallest n_modes >= k that does not cut a cluster of (numerically) equal eigenvalues."""
    for g in modal.clusters(lam_all, 1e-6):
        if g[0] < k <= g[-1]:
            k = g[-1] + 1
    return k


@pytest.mark.parametrize("consistent", [False, True], ids=["lumped", "consistent"])
@pytest.mark.parametrize("name", [f[0] for f in fixtures()])
def test_fixtures_against_oracle(name, consistent):
    dim, joints, support, conn, aed = arrays(name)
    plan = _lib.Plan(dim, conn, support)
    assert plan.n <= 160
    for jm in (None, joint_masses(dim, joints, conn, aed)):
        lam_all = modal.modes(dim, joints, support, conn, aed, consistent=consistent, joint_mass=jm)["eigval_all"]
        for k in sorted({plan.n, uncut(lam_all, min(10, plan.n))}):
            out = plan.modes_host(1, joints, aed=aed, n_modes=k, consistent=consistent, joint_mass=jm)
            assert out["info"][0] == 0
            check_against_oracle(dim, joints, support, conn, aed, out["eigval"][0], out["modes"][0], consistent, jm)


@pytest.mark.parametrize("name", ["bar-72_input_0", "bar-120_input_0"])
def test_cut_cluster_still_accurate(name):
    dim, joints, support, conn, aed = arrays(name)
    plan = _lib.Plan(dim, conn, support)
    lam_all = modal.modes(dim, joints, support, conn, aed)["eigval_all"]
    cl = [g for g in modal.clusters(lam_all, 1e-9) if len(g) > 1 and g[0] < 20]
    assert cl, "the fixture has repeated frequencies among its lowest modes"
    k = cl[0][0] + 1                                      # keeps one vector of the pair
    out = plan.modes_host(1, joints, aed=aed, n_modes=k)
    assert out["info"][0] == 0
    ref = modal.modes(dim, joints, support, conn, aed)
    lmax = np.abs(lam_all).max()
    assert np.abs(out["eigval"][0] - lam_all[:k]).max() <= TOL_VAL * lmax
    phi = out["modes"][0][:, ref["mask"]].T
    Mphi = ref["M_ff"] @ phi
    assert np.abs(ref["K_ff"] @ phi - Mphi * out["eigval"][0]).max() <= TOL_VAL * lmax * np.abs(Mphi).max()


def perturbed(aed, B, seed, spread=0.3):
    rng = np.random.default_rng(seed)
    return np.stack([aed * rng.uniform(1 - spread, 1 + spread, size=aed.shape) for _ in range(B)])


def device_modes(plan, B, xyz, aed=None, gene=None, table=None, **kw):
    import torch

    dev = torch.device("cuda:0")
    td = lambda a, dt=torch.float64: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(dev, dt)  # noqa: E731
    k = plan.n if kw.get("n_modes") is None else kw["n_modes"]
    out = {"modes": torch.empty(B, k, plan.N, dtype=torch.float64, device=dev)}
    jm = kw.pop("joint_mass", None)
    plan.modes_device(B, td(xyz), aed=td(aed), gene=td(gene, torch.int32), type_table=td(table), joint_mass=td(jm), out=out,
                      **kw)
    torch.cuda.synchronize()
    return {k2: v.cpu().numpy() for k2, v in out.items()}


@pytest.mark.parametrize("consistent", [False, True], ids=["lumped", "consistent"])
def test_bits_do_not_depend_on_the_launch(consistent):
    dim, joints, support, conn, aed = arrays("bar-72_input_0")
    plan = _lib.Plan(dim, conn, support)
    B = 5000                                              # more systems than resident CTAs: the grid-stride loop runs
    A = perturbed(aed, B, 1)
    jm = joint_masses(dim, joints, conn, aed)
    big = device_modes(plan, B, joints, aed=A, n_modes=12, consistent=consistent, joint_mass=jm)
    assert np.all(big["info"] == 0)
    for b in (0, 1, 777, B - 1):
        solo = plan.modes_host(1, joints, aed=A[b], n_modes=12, consistent=consistent, joint_mass=jm)
        assert np.array_equal(solo["eigval"][0], big["eigval"][b]) and np.array_equal(solo["modes"][0], big["modes"][b])
    mid = device_modes(plan, 300, joints, aed=A[700:1000], n_modes=12, consistent=consistent, joint_mass=jm)
    assert np.array_equal(mid["eigval"], big["eigval"][700:1000]) and np.array_equal(mid["modes"], big["modes"][700:1000])
    # stride-0 shared inputs == the same rows repeated
    rep = device_modes(plan, 40, np.tile(joints.reshape(-1), (40, 1)), aed=np.tile(A[5].reshape(-1), (40, 1)), n_modes=12,
                       consistent=consistent, joint_mass=np.tile(jm, (40, 1)))
    sh = device_modes(plan, 40, joints, aed=A[5], n_modes=12, consistent=consistent, joint_mass=jm)
    assert np.array_equal(rep["eigval"], sh["eigval"]) and np.array_equal(rep["modes"], sh["modes"])
    assert np.array_equal(sh["eigval"][3], big["eigval"][5])
    # n_modes = k gives the first k of n_modes = n
    full = device_modes(plan, 64, joints, aed=A[:64], consistent=consistent, joint_mass=jm)
    assert np.array_equal(full["eigval"][:, :12], big["eigval"][:64]) and np.array_equal(full["modes"][:, :12], big["modes"][:64])


def test_gene_table_equals_expanded_aed():
    dim, joints, support, conn, aed = arrays("bar-72_input_0")
    plan = _lib.Plan(dim, conn, support)
    rng = np.random.default_rng(3)
    table = np.stack([rng.uniform(0.5, 3.0, 8), rng.uniform(1e7, 3e7, 8), rng.uniform(0.05, 0.3, 8)], 1)
    genes = rng.integers(0, 8, size=(500, plan.M)).astype(np.int32)
    for consistent in (False, True):
        g = device_modes(plan, 500, joints, gene=genes, table=table, n_modes=6, consistent=consistent)
        a = device_modes(plan, 500, joints, aed=table[genes], n_modes=6, consistent=consistent)
        assert np.all(g["info"] == 0)
        assert np.array_equal(g["eigval"], a["eigval"]) and np.array_equal(g["modes"], a["modes"])
        h = plan.modes_host(500, joints, gene=genes, type_table=table, n_modes=6, consistent=consistent)
        assert np.array_equal(h["eigval"], a["eigval"]) and np.array_equal(h["modes"], a["modes"])


@pytest.mark.parametrize("consistent", [False, True], ids=["lumped", "consistent"])
def test_failures_share_ctas_with_good_systems(consistent):
    dim, joints, support, conn, aed = arrays("bar-72_input_0")
    plan = _lib.Plan(dim, conn, support)
    B = 3000
    A = perturbed(aed, B, 7)
    X = np.tile(joints, (B, 1, 1))
    want = {}
    X[11, conn[4, 1]] = X[11, conn[4, 0]]                     # zero-length member
    want[11] = -2
    free_joint = int(np.nonzero(support == orc.NO)[0][0])
    for b in (12, 1500, 2999):                                 # no mass at a free joint
        A[b, (conn == free_joint).any(axis=1), 2] = 0.0
        want[b] = _lib.TB_INFO_MASS
    out = device_modes(plan, B, X, aed=A, n_modes=8, consistent=consistent)
    for b in range(B):
        assert out["info"][b] == want.get(b, 0), b
    for b in want:
        assert not out["eigval"][b].any() and not out["modes"][b].any()
    for b in (10, 13, 1499, 2998):
        solo = plan.modes_host(1, joints, aed=A[b], n_modes=8, consistent=consistent)
        assert np.array_equal(solo["eigval"][0], out["eigval"][b]) and np.array_equal(solo["modes"][0], out["modes"][b])
    # a gene out of range
    table = aed[:3].copy()
    genes = np.zeros((200, plan.M), np.int32)
    genes[50, 3] = 3
    g = device_modes(plan, 200, joints, gene=genes, table=table, n_modes=8, consistent=consistent)
    assert g["info"][50] == -4 and not g["eigval"][50].any() and not g["modes"][50].any()
    assert np.all(np.delete(g["info"], 50) == 0)
    assert np.array_equal(g["eigval"][49], g["eigval"][51])


@pytest.mark.parametrize("consistent", [False, True], ids=["lumped", "consistent"])
def test_counting_rule_and_mechanism(consistent):
    # counting rule: a 2D triangle with one pin and nothing else (3 + 2 < 6)
    j = np.array([[0.0, 0.0], [4.0, 0.0], [2.0, 3.0]])
    plan = _lib.Plan(2, np.array([[0, 1], [1, 2], [0, 2]], np.int32), np.array([orc.PIN, 0, 0], np.uint8))
    out = plan.modes_host(5, j, aed=np.tile([1.0, 1e7, 0.1], (3, 1)), n_modes=2, consistent=consistent)
    assert np.all(out["info"] == -1) and not out["eigval"].any() and not out["modes"].any()
    # a sway mechanism that passes the counting rule (the member between the two pins adds no stiffness to K_ff)
    j = np.array([[0.0, 0.0], [1.0, 0.0], [1.0, 1.0], [0.0, 1.0]])
    conn = np.array([[0, 3], [1, 2], [2, 3], [0, 1]], np.int32)
    sup = np.array([orc.PIN, orc.PIN, 0, 0], np.uint8)
    plan = _lib.Plan(2, conn, sup)
    assert plan.stable
    aed = np.tile([1.0, 1e7, 0.1], (4, 1))
    out = plan.modes_host(1, j, aed=aed, consistent=consistent)
    assert out["info"][0] == 0
    lam = out["eigval"][0]
    assert abs(lam[0]) <= TOL_VAL * lam.max()


def test_consistent_scratch_in_a_cuda_graph():
    import torch

    dim, joints, support, conn, aed = arrays("bar-72_input_0")
    dev = torch.device("cuda:0")
    td = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(dev)  # noqa: E731
    A = perturbed(aed, 600, 5)
    plan = _lib.Plan(dim, conn, support)
    xyz, aedt = td(joints), td(A)
    out = {"eigval": torch.empty(600, 6, dtype=torch.float64, device=dev), "info": torch.empty(600, dtype=torch.int32, device=dev),
           "modes": torch.empty(600, 6, plan.N, dtype=torch.float64, device=dev)}
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        plan.modes_device(600, xyz, aed=aedt, n_modes=6, consistent=True, out=out, stream=s)   # warm-up: grows the slots
    s.synchronize()
    want = {k: v.clone() for k, v in out.items()}
    for v in out.values():
        v.zero_()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        plan.modes_device(600, xyz, aed=aedt, n_modes=6, consistent=True, out=out, stream=s)
    g.replay()
    torch.cuda.synchronize()
    for k in want:
        assert torch.equal(out[k], want[k])
    # a fresh plan has no slots: a captured call would have to grow them -> TB_ERR_ALLOC, nothing enqueued
    fresh = _lib.Plan(dim, conn, support)
    out2 = {"eigval": torch.full((600, 6), 7.0, dtype=torch.float64, device=dev), "info": torch.full((600,), 7, dtype=torch.int32, device=dev)}
    g2 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g2, stream=s):
        with pytest.raises(_lib.TrussLibError) as e:
            fresh.modes_device(600, xyz, aed=aedt, n_modes=6, consistent=True, out=out2, stream=s)
        out2["eigval"].add_(0.0)                           # (keeps the captured graph non-empty)
    assert e.value.code == _lib.TB_ERR_ALLOC
    g2.replay()
    torch.cuda.synchronize()
    assert bool((out2["info"] == 7).all()) and bool((out2["eigval"] == 7.0).all())
    # lumped mass needs no scratch: capturable on a fresh plan
    g3 = torch.cuda.CUDAGraph()
    out3 = {"eigval": torch.empty(600, 6, dtype=torch.float64, device=dev), "info": torch.empty(600, dtype=torch.int32, device=dev)}
    with torch.cuda.graph(g3, stream=s):
        fresh.modes_device(600, xyz, aed=aedt, n_modes=6, out=out3, stream=s)
    g3.replay()
    torch.cuda.synchronize()
    ref = plan.modes_host(600, joints, aed=A, n_modes=6, want_modes=False)
    assert np.array_equal(out3["eigval"].cpu().numpy(), ref["eigval"])


def test_one_native_launch_per_call():
    import torch

    dim, joints, support, conn, aed = arrays("bar-10_input_0")
    plan = _lib.Plan(dim, conn, support)
    dev = torch.device("cuda:0")
    x, a = torch.from_numpy(joints.copy()).to(dev), torch.from_numpy(aed.copy()).to(dev)
    for consistent in (False, True):
        n0 = _lib.launch_count()
        out = plan.modes_device(4, x, aed=a, n_modes=3, consistent=consistent)
        torch.cuda.synchronize()
        assert _lib.launch_count() - n0 == 1                # one k_modes launch, nothing else
        assert not out["info"].any() and bool((out["eigval"] > 0).all())


def test_python_api():
    from python_stable_3d_truss_analysis_b200.batch import ModesBatch
    from python_stable_3d_truss_analysis_b200.truss import MassNotPositiveDefiniteError, Truss
    from python_stable_3d_truss_analysis_b200.type import MemberType

    data = H.load_json("ref_data/bar-72_input_0.json")
    t = Truss(3).LoadFromJSON(data=data)
    dim, joints, support, conn, aed = arrays("bar-72_input_0")
    jm = {3: 2.5, 7: 1.0}
    jarr = np.zeros(len(joints))
    for k, v in jm.items():
        jarr[k] = v
    t.SolveModes(nMode=12, jointMasses=jm)
    ref = modal.modes(dim, joints, support, conn, aed, joint_mass=jarr)
    lam = t.GetEigenvalues()
    assert np.abs(lam - ref["eigval_all"][:12]).max() <= TOL_VAL * ref["eigval_all"].max()
    assert np.array_equal(t.GetNaturalFrequencies(), np.sqrt(lam) / (2 * np.pi))
    shapes = t.GetModeShapes()
    assert len(shapes) == 12 and set(shapes[0]) == set(range(t.nJoint))
    dense = np.stack([np.concatenate([s[j] for j in range(t.nJoint)]) for s in shapes])
    check_against_oracle(dim, joints, support, conn, aed, lam, dense, False, jarr)
    t.SetJointPosition(5, tuple(np.asarray(t.GetJointPosition(5)) + 1.0))
    with pytest.raises(Exception):
        t.GetEigenvalues()
    # a GA population: ModesBatch == per-design SolveModes
    types = [MemberType(*row) for row in np.unique(aed, axis=0)] + [MemberType(2.0, 1e7, 0.1), MemberType(0.5, 1e7, 0.1)]
    rng = np.random.default_rng(9)
    genes = rng.integers(0, len(types), size=(64, t.nMember)).astype(np.int32)
    t = Truss(3).LoadFromJSON(data=data)
    pop = ModesBatch(t, genes=genes, memberTypeList=types, nMode=6, isConsistentMass=True)
    for b in (0, 31, 63):
        for m, g in enumerate(genes[b]):
            t.SetMemberType(m, types[g])
        t.SolveModes(nMode=6, isConsistentMass=True)
        assert np.array_equal(t.GetEigenvalues(), pop["eigval"][b])
    zero = aed.copy()
    zero[:, 2] = 0.0
    with pytest.raises(MassNotPositiveDefiniteError):
        ModesBatch(t, aed=zero[None], nMode=3)
