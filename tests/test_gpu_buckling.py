"""Linear buckling on the GPU (tb_buckling / tb_buckling_host, k_buckling<DIM>) with the member forces of tb_solve on the
same batch: load factors and buckling modes against the numpy oracle (oracle/buckling.py) on every fixture up to 160
free DOFs and the braced column's closed form; bit invariance under batch position, batch size, strides, gene tables,
n_modes and the entry point; failures among good systems; the modal arena under CUDA graph capture; and the Python API."""
import numpy as np
import pytest

from oracle import buckling as bk
from oracle import modal
from oracle import truss_oracle as orc
from python_stable_3d_truss_analysis_b200 import _lib
from tests import helpers as H
from tests.test_buckling_cpu import braced_column

pytestmark = pytest.mark.gpu

TOL_VAL = 1e-11      # |nu - nu_ref| <= TOL_VAL * max|nu| and the residual
TOL_ORTH = 1e-10     # K-orthonormality
TOL_VEC = 1e-8       # isolated vectors and cluster projectors
CLEAR = 1e-6         # nu < -CLEAR * max|nu|: clearly critical, compared with the oracle


def fixtures():
    return [(n, d, data) for n, d, data, _ in H.shipped_cases() if not n.startswith("bar-942")] + \
        [(n, d, data) for n, d, data, _ in H.cube7_shipped()[:2]]


def arrays(name):
    for n, d, data in fixtures():
        if n == name:
            return (d,) + tuple(orc.arrays_from_json(data, d))
    raise KeyError(name)


def check_against_oracle(dim, joints, support, conn, aed, axial, got_fac, got_vec):
    """Every check of one system against the oracle fed the same member forces."""
    ref = bk.buckling(dim, joints, support, conn, aed, axial)
    K, KG, mask, nu = ref["K_ff"], ref["K_G_ff"], ref["mask"], ref["nu"]
    k = len(got_fac)
    numax = np.abs(nu).max()
    fin = np.isfinite(got_fac)
    assert np.all(got_fac[fin] > 0) and np.all(np.diff(got_fac[fin]) >= 0)
    assert np.all(fin[:-1] >= fin[1:])                     # the finite factors come first
    clear = nu[:k] < -CLEAR * numax
    assert np.all(fin[clear])
    assert np.all(~fin[nu[:k] > CLEAR * numax])
    assert np.abs(-1.0 / got_fac[clear] - nu[:k][clear]).max(initial=0.0) <= TOL_VAL * numax
    assert np.all(got_vec[:, ~mask] == 0.0) and np.all(got_vec[~fin] == 0.0)
    phi = got_vec[fin][:, mask].T                          # [n, k_fin]
    if phi.size:
        lam = got_fac[fin]
        Kphi = K @ phi
        res = Kphi + (KG @ phi) * lam                      # = lambda (K_G phi - nu K phi)
        assert np.all(np.abs(res).max(axis=0) <= TOL_VAL * lam * numax * np.abs(Kphi).max(axis=0))
        assert np.abs(phi.T @ Kphi - np.eye(phi.shape[1])).max() <= TOL_ORTH
        big = np.argmax(np.abs(phi), axis=0)
        assert np.all(phi[big, np.arange(phi.shape[1])] > 0)
    ref_phi = ref["modes"][:k][:, mask].T
    ncl = int(clear.sum())
    for g in modal.clusters(nu, CLEAR):
        if g[-1] >= ncl:                                   # (only clusters of clearly critical modes, not cut by k)
            continue
        if len(g) == 1:
            a, b = phi[:, g[0]], ref_phi[:, g[0]]
            mags = np.sort(np.abs(b))[::-1]
            if len(mags) > 1 and mags[0] - mags[1] <= 1e-8 * mags[0]:
                b = b * np.sign(a @ K @ b)                  # a near tie of the largest components: the sign is rounding's
            assert np.linalg.norm(a - b) <= TOL_VEC * np.linalg.norm(b)
        else:                                              # a cluster: its K-projector
            P = phi[:, g] @ phi[:, g].T @ K
            Pr = ref_phi[:, g] @ ref_phi[:, g].T @ K
            assert np.abs(P - Pr).max() <= TOL_VEC * max(1.0, np.abs(Pr).max())
    return int(fin.sum())


def static_axial(plan, B, xyz, force, **props):
    out = plan.solve_host(B, xyz, force, want=("axial",), **props)
    assert np.all(out["info"] == 0)
    return out["axial"]


@pytest.mark.parametrize("name", [f[0] for f in fixtures()])
def test_fixtures_against_oracle(name):
    dim, joints, support, conn, aed, force = arrays(name)
    plan = _lib.Plan(dim, conn, support)
    assert plan.n <= 160
    ax = static_axial(plan, 1, joints, force, aed=aed)[0]
    for k in sorted({plan.n, min(6, plan.n)}):
        out = plan.buckling_host(1, joints, ax, aed=aed, n_modes=k)
        assert out["info"][0] == 0
        nfin = check_against_oracle(dim, joints, support, conn, aed, ax, out["factor"][0], out["modes"][0])
        assert nfin >= 1


@pytest.mark.parametrize("dim", [2, 3])
def test_braced_column_closed_form(dim):
    Es, As, L, b, P = 3.0e7, 0.25, 4.0, 3.0, 1.0e3
    joints, support, conn, aed, force = braced_column(dim, Es=Es, As=As, L=L, b=b, P=P)
    plan = _lib.Plan(dim, conn, support)
    ax = static_axial(plan, 1, joints, force, aed=aed)[0]
    out = plan.buckling_host(1, joints, ax, aed=aed)
    assert out["info"][0] == 0
    fac, modes = out["factor"][0], out["modes"][0]
    nfin = dim - 1
    assert np.allclose(fac[:nfin], Es * As * L / (b * P), rtol=1e-12, atol=0)
    assert np.all(np.isinf(fac[nfin:])) and np.all(modes[nfin:] == 0.0)
    if dim == 2:
        assert np.allclose(modes[0], [0, 0, 1 / np.sqrt(Es * As / b), 0, 0, 0], rtol=1e-12, atol=0)
    else:
        phi = modes[:2][:, 3:5]
        assert np.allclose(phi @ phi.T, np.eye(2) / (Es * As / b), rtol=1e-12, atol=1e-20)
    # the reversed load never buckles; zero forces are not an error
    for state in (-ax, 0.0 * ax):
        out = plan.buckling_host(1, joints, state, aed=aed)
        assert out["info"][0] == 0 and np.all(np.isinf(out["factor"][0])) and not out["modes"].any()


def perturbed(aed, B, seed, spread=0.3):
    rng = np.random.default_rng(seed)
    return np.stack([aed * rng.uniform(1 - spread, 1 + spread, size=aed.shape) for _ in range(B)])


def td(a, dt=None):
    import torch

    if a is None:
        return None
    return torch.from_numpy(np.ascontiguousarray(a)).to(torch.device("cuda:0"), dt or torch.float64)


def device_buckling(plan, B, xyz, axial, aed=None, gene=None, table=None, **kw):
    import torch

    k = plan.n if kw.get("n_modes") is None else kw["n_modes"]
    out = {"modes": torch.empty(B, k, plan.N, dtype=torch.float64, device="cuda:0")}
    plan.buckling_device(B, td(xyz), td(axial), aed=td(aed), gene=td(gene, torch.int32), type_table=td(table), out=out,
                         **kw)
    torch.cuda.synchronize()
    return {k2: v.cpu().numpy() for k2, v in out.items()}


def device_axial(plan, B, xyz, force, aed):
    import torch

    out = {"axial": torch.empty(B, plan.M, dtype=torch.float64, device="cuda:0"),
           "info": torch.empty(B, dtype=torch.int32, device="cuda:0")}
    plan.solve_device(B, td(xyz), td(force), aed=td(aed), out=out)
    torch.cuda.synchronize()
    return out["axial"].cpu().numpy(), out["info"].cpu().numpy()


def same(a, b):
    return np.array_equal(a["factor"], b["factor"]) and np.array_equal(a["modes"], b["modes"]) and \
        np.array_equal(a["info"], b["info"])


def test_bits_do_not_depend_on_the_launch():
    dim, joints, support, conn, aed, force = arrays("bar-72_input_0")
    plan = _lib.Plan(dim, conn, support)
    B = 5000                                              # more systems than resident CTAs: the grid-stride loop runs
    A = perturbed(aed, B, 1)
    AX, info = device_axial(plan, B, joints, force, A)
    assert np.all(info == 0)
    big = device_buckling(plan, B, joints, AX, aed=A, n_modes=12)
    assert np.all(big["info"] == 0) and np.isfinite(big["factor"][:, 0]).all()
    for b in (0, 1, 777, B - 1):                           # device == host entry point, batch of one
        solo = plan.buckling_host(1, joints, AX[b], aed=A[b], n_modes=12)
        assert np.array_equal(solo["factor"][0], big["factor"][b]) and np.array_equal(solo["modes"][0], big["modes"][b])
    mid = device_buckling(plan, 300, joints, AX[700:1000], aed=A[700:1000], n_modes=12)
    assert np.array_equal(mid["factor"], big["factor"][700:1000]) and np.array_equal(mid["modes"], big["modes"][700:1000])
    # stride-0 shared inputs (axial included) == the same rows repeated
    rep = device_buckling(plan, 40, np.tile(joints.reshape(-1), (40, 1)), np.tile(AX[5], (40, 1)),
                          aed=np.tile(A[5].reshape(-1), (40, 1)), n_modes=12)
    sh = device_buckling(plan, 40, joints, AX[5], aed=A[5], n_modes=12)
    assert same(rep, sh)
    assert np.array_equal(sh["factor"][3], big["factor"][5]) and np.array_equal(sh["modes"][3], big["modes"][5])
    # an explicit axial stride: every other row of a [2B, M] array
    wide = np.zeros((80, plan.M))
    wide[::2] = AX[:40]
    st = device_buckling(plan, 40, joints, wide, aed=A[:40], n_modes=12, axial_stride=2 * plan.M)
    assert np.array_equal(st["factor"], big["factor"][:40]) and np.array_equal(st["modes"], big["modes"][:40])
    # n_modes = k gives the first k of n_modes = n
    full = device_buckling(plan, 64, joints, AX[:64], aed=A[:64])
    assert np.array_equal(full["factor"][:, :12], big["factor"][:64]) and np.array_equal(full["modes"][:, :12], big["modes"][:64])
    # the host entry point on the whole batch
    host = plan.buckling_host(B, joints, AX, aed=A, n_modes=12)
    assert same(host, big)


def test_gene_table_equals_expanded_aed():
    dim, joints, support, conn, aed, force = arrays("bar-72_input_0")
    plan = _lib.Plan(dim, conn, support)
    rng = np.random.default_rng(3)
    table = np.stack([rng.uniform(0.5, 3.0, 8), rng.uniform(1e7, 3e7, 8), rng.uniform(0.05, 0.3, 8)], 1)
    genes = rng.integers(0, 8, size=(500, plan.M)).astype(np.int32)
    AX = static_axial(plan, 500, joints, force, gene=genes, type_table=table)
    g = device_buckling(plan, 500, joints, AX, gene=genes, table=table, n_modes=6)
    a = device_buckling(plan, 500, joints, AX, aed=table[genes], n_modes=6)
    assert np.all(g["info"] == 0)
    assert same(g, a)
    h = plan.buckling_host(500, joints, AX, gene=genes, type_table=table, n_modes=6)
    assert same(h, a)


def test_host_validates_the_axial_stride():
    dim, joints, support, conn, aed, force = arrays("bar-72_input_0")
    plan = _lib.Plan(dim, conn, support)
    with pytest.raises(_lib.TrussLibError) as e:
        plan.buckling_host(2, joints, np.zeros((2, plan.M + 1)), aed=aed, n_modes=6, axial_stride=plan.M + 1)
    assert e.value.code == -3


def test_failures_share_ctas_with_good_systems():
    dim, joints, support, conn, aed, force = arrays("bar-72_input_0")
    plan = _lib.Plan(dim, conn, support)
    B = 3000
    A = perturbed(aed, B, 7)
    X = np.tile(joints, (B, 1, 1))
    want = {}
    X[11, conn[4, 1]] = X[11, conn[4, 0]]                     # zero-length member
    want[11] = -2
    free_joint = int(np.nonzero(support == orc.NO)[0][0])
    mech = (12, 1500, 2999)
    for b in mech:                                            # no stiffness at a free joint: a mechanism
        A[b, (conn == free_joint).any(axis=1), 1] = 0.0
    AX, sinfo = device_axial(plan, B, X, force, A)
    assert sinfo[11] == -2 and all(sinfo[b] > 0 for b in mech)
    assert np.count_nonzero(sinfo) == 1 + len(mech)
    AX[20] = 0.0                                              # zero forces: all factors inf, info 0
    out = device_buckling(plan, B, X, AX, aed=A, n_modes=8)
    for b in range(B):
        if b in mech:
            assert out["info"][b] > 0, b                      # K_ff is not positive definite, as for tb_solve
        else:
            assert out["info"][b] == want.get(b, 0), b
    for b in list(want) + list(mech):
        assert not out["factor"][b].any() and not out["modes"][b].any()
    assert np.all(np.isinf(out["factor"][20])) and not out["modes"][20].any()
    for b in (10, 13, 1499, 2998):
        solo = plan.buckling_host(1, joints, AX[b], aed=A[b], n_modes=8)
        assert np.array_equal(solo["factor"][0], out["factor"][b]) and np.array_equal(solo["modes"][0], out["modes"][b])
    # a gene out of range
    table = aed[:3].copy()
    genes = np.zeros((200, plan.M), np.int32)
    genes[50, 3] = 3
    ax = static_axial(plan, 1, joints, force, aed=table[genes[0]])
    g = device_buckling(plan, 200, joints, ax[0], gene=genes, table=table, n_modes=8)
    assert g["info"][50] == -4 and not g["factor"][50].any() and not g["modes"][50].any()
    assert np.all(np.delete(g["info"], 50) == 0)
    assert np.array_equal(g["factor"][49], g["factor"][51])


def test_counting_rule_and_mechanism():
    # counting rule: a 2D triangle with one pin and nothing else (3 + 2 < 6)
    j = np.array([[0.0, 0.0], [4.0, 0.0], [2.0, 3.0]])
    plan = _lib.Plan(2, np.array([[0, 1], [1, 2], [0, 2]], np.int32), np.array([orc.PIN, 0, 0], np.uint8))
    out = plan.buckling_host(5, j, np.full(3, -1.0), aed=np.tile([1.0, 1e7, 0.1], (3, 1)), n_modes=2)
    assert np.all(out["info"] == -1) and not out["factor"].any() and not out["modes"].any()
    # a joint between two pins on a straight line passes the counting rule; K_ff has a zero row (its y DOF)
    j = np.array([[0.0, 0.0], [1.0, 0.0], [2.0, 0.0]])
    plan = _lib.Plan(2, np.array([[0, 1], [1, 2]], np.int32), np.array([orc.PIN, 0, orc.PIN], np.uint8))
    assert plan.stable
    aed = np.tile([1.0, 1e7, 0.1], (2, 1))
    st = plan.solve_host(1, j, np.zeros(6), aed=aed)
    out = plan.buckling_host(1, j, np.array([-1.0, -1.0]), aed=aed)
    assert st["info"][0] > 0 and out["info"][0] == 2        # the pivot of free DOF 1 (y of joint 1)
    assert not out["factor"].any() and not out["modes"].any()


def test_arena_in_a_cuda_graph():
    import torch

    dim, joints, support, conn, aed, force = arrays("bar-72_input_0")
    dev = torch.device("cuda:0")
    A = perturbed(aed, 600, 5)
    plan = _lib.Plan(dim, conn, support)
    AX = static_axial(plan, 600, joints, force, aed=A)
    xyz, aedt, axt = td(joints), td(A), td(AX)
    out = {"factor": torch.empty(600, 6, dtype=torch.float64, device=dev), "info": torch.empty(600, dtype=torch.int32, device=dev),
           "modes": torch.empty(600, 6, plan.N, dtype=torch.float64, device=dev)}
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        plan.buckling_device(600, xyz, axt, aed=aedt, n_modes=6, out=out, stream=s)   # warm-up: grows the arena
    s.synchronize()
    want = {k: v.clone() for k, v in out.items()}
    for v in out.values():
        v.zero_()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        plan.buckling_device(600, xyz, axt, aed=aedt, n_modes=6, out=out, stream=s)
    g.replay()
    torch.cuda.synchronize()
    for k in want:
        assert torch.equal(out[k], want[k])
    # a fresh plan has no arena: a captured call would have to grow it -> TB_ERR_ALLOC, nothing enqueued
    fresh = _lib.Plan(dim, conn, support)
    out2 = {"factor": torch.full((600, 6), 7.0, dtype=torch.float64, device=dev),
            "info": torch.full((600,), 7, dtype=torch.int32, device=dev)}
    g2 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g2, stream=s):
        with pytest.raises(_lib.TrussLibError) as e:
            fresh.buckling_device(600, xyz, axt, aed=aedt, n_modes=6, out=out2, stream=s)
        out2["factor"].add_(0.0)                           # (keeps the captured graph non-empty)
    assert e.value.code == _lib.TB_ERR_ALLOC
    g2.replay()
    torch.cuda.synchronize()
    assert bool((out2["info"] == 7).all()) and bool((out2["factor"] == 7.0).all())


def test_one_native_launch_per_call():
    import torch

    dim, joints, support, conn, aed, force = arrays("bar-10_input_0")
    plan = _lib.Plan(dim, conn, support)
    ax = static_axial(plan, 1, joints, force, aed=aed)[0]
    x, a, n = td(joints), td(aed), td(ax)
    plan.buckling_device(4, x, n, aed=a, n_modes=3)           # (the arena grows on the first call)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    out = plan.buckling_device(4, x, n, aed=a, n_modes=3)
    torch.cuda.synchronize()
    assert _lib.launch_count() - n0 == 1                    # one k_buckling launch, nothing else
    assert not out["info"].any() and bool((out["factor"][:, 0] > 0).all())


def test_python_api():
    from python_stable_3d_truss_analysis_b200.batch import BucklingBatch
    from python_stable_3d_truss_analysis_b200.truss import Truss
    from python_stable_3d_truss_analysis_b200.type import MemberType

    data = H.load_json("ref_data/bar-72_input_0.json")
    t = Truss(3).LoadFromJSON(data=data)
    dim, joints, support, conn, aed, force = arrays("bar-72_input_0")
    t.SolveBuckling(nMode=12)
    plan = _lib.Plan(dim, conn, support)
    ax = static_axial(plan, 1, joints, force, aed=aed)[0]
    fac = t.GetBucklingFactors()
    shapes = t.GetBucklingModes()
    assert len(fac) == 12 and len(shapes) == 12 and set(shapes[0]) == set(range(t.nJoint))
    dense = np.stack([np.concatenate([s[j] for j in range(t.nJoint)]) for s in shapes])
    check_against_oracle(dim, joints, support, conn, aed, ax, fac, dense)
    t.SetMemberType(0, MemberType(2.0, 1e7, 0.1))
    with pytest.raises(Exception):
        t.GetBucklingFactors()
    t = Truss(3).LoadFromJSON(data=data)
    t.SolveBuckling(nMode=4)
    t.AddExternalForce(5, (1.0, 0.0, 0.0))
    with pytest.raises(Exception):
        t.GetBucklingModes()
    # a GA population of 8192 designs: one static call and one buckling launch, the oracle on a sample
    types = [MemberType(*row) for row in np.unique(aed, axis=0)] + [MemberType(2.0, 1e7, 0.1), MemberType(0.5, 1e7, 0.1)]
    table = np.array([m.Serialize() for m in types])
    rng = np.random.default_rng(9)
    genes = rng.integers(0, len(types), size=(8192, t.nMember)).astype(np.int32)
    t = Truss(3).LoadFromJSON(data=data)
    BucklingBatch(t, genes=genes[:2], memberTypeList=types, nMode=6)   # (warm: plan and arenas)
    n0 = _lib.launch_count()
    t._get_plan().solve_host(8192, joints, force, gene=genes, type_table=table, want=("axial",))
    n_static = _lib.launch_count() - n0
    n0 = _lib.launch_count()
    pop = BucklingBatch(t, genes=genes, memberTypeList=types, nMode=6)
    assert _lib.launch_count() - n0 == n_static + 1
    assert np.all(pop["info"] == 0) and pop["factor"].shape == (8192, 6) and pop["modes"].shape == (8192, 6, t.nJoint * 3)
    for b in (0, 4095, 8191):
        a_b = table[genes[b]]
        assert np.abs(pop["axial"][b] - orc.solve(dim, joints, support, conn, a_b, force)["axial"]).max() <= \
            1e-9 * np.abs(pop["axial"][b]).max()
        check_against_oracle(dim, joints, support, conn, a_b, pop["axial"][b], pop["factor"][b], pop["modes"][b])
    for b in (0, 8191):                                     # == Truss.SolveBuckling per design
        for m, g in enumerate(genes[b]):
            t.SetMemberType(m, types[g])
        t.SolveBuckling(nMode=6)
        assert np.array_equal(t.GetBucklingFactors(), pop["factor"][b])
