"""Parity of the CUDA path (through the C ABI) against the reference's golden files, the
live-reference vectors and the oracle.  Tolerance: 1e-9 norm-wise per field (north_star);
index maps are checked bit-exact in tests/test_abi_cpu.py."""
import ctypes as C
import json

import numpy as np
import pytest

from oracle import truss_oracle as orc
from python_stable_3d_truss_analysis_b200 import _lib
from python_stable_3d_truss_analysis_b200.batch import (FitnessBatch, SolveBatch, SolveLoadCases, SolveMemberTypes,
                                                          type_table)
from python_stable_3d_truss_analysis_b200.truss import Truss
from python_stable_3d_truss_analysis_b200.type import MemberType, SupportType
from python_stable_3d_truss_analysis_b200.utils import TrussNotStableError
from tests import band_catalogue as BC
from tests import helpers as H
from tests.helpers import tower as _tower

pytestmark = pytest.mark.gpu


def dense(t):
    return {"u": t._dense["u"], "ext": t._dense["ext"], "axial": t._dense["axial"], "weight": t.weight}


PATHS = pytest.mark.parametrize("path", [0, 1, 2], ids=["fused", "tiled", "band"])


def force_path(plan, path):
    try:
        plan.set_path(path)
    except _lib.TrussLibError as exc:
        if exc.code == _lib.TB_ERR_TOO_LARGE:
            pytest.skip("system does not fit this pipeline")
        raise


@PATHS
@pytest.mark.parametrize("name,dim,data,gold", H.shipped_cases(), ids=lambda v: v if isinstance(v, str) else None)
def test_solve_vs_shipped_goldens(name, dim, data, gold, path):
    t = Truss(dim).LoadFromJSON(data=data)
    plan = t._get_plan()
    force_path(plan, path)
    t.Solve()
    H.assert_close(dense(t), gold, what=f"{name} path{path}")
    for k in H.FIELDS:
        assert H.key_sets_match(t._dense[k], gold[k]), (name, k)
    # sparse dict views follow the 1e-10 filter
    for j, v in t.GetDisplacements().items():
        assert not (np.abs(v) < 1e-10).all()
    ser = t.Serialize()
    assert set(ser) >= {"displace", "external", "internal", "weight"}


@pytest.mark.parametrize("name,dim,data,gold", H.cube7_shipped(), ids=lambda v: v if isinstance(v, str) else None)
def test_solve_vs_shipped_cube7(name, dim, data, gold):
    t = Truss(dim).LoadFromJSON(data=data)
    t.Solve()
    H.assert_close(dense(t), gold, what=name)


@PATHS
def test_solve_vs_live_random(path):
    for i, case in enumerate(H.load_json("live_random.json")):
        dim = case["dim"]
        t = Truss(dim).LoadFromJSON(data=case["data"])
        force_path(t._get_plan(), path)
        t.Solve()
        want = {k: np.array(v) if k != "weight" else v for k, v in case["result"].items()}
        H.assert_close(dense(t), want, what=f"random[{i}] path{path}")


def test_ragged_batch_vs_live_cube7_aug():
    live = H.load_json("live_cube7_aug.json")
    trusses = [Truss(3).LoadFromJSON(data=g) for g in live]
    assert len({(t.nJoint, t.nMember) for t in trusses}) > 1          # genuinely ragged
    info = SolveBatch(trusses)
    assert not info.any()
    for i, (t, g) in enumerate(zip(trusses, live)):
        H.assert_close(dense(t), H.dense_from_output(g, 3), what=f"cube7_aug[{i}]")


def test_uniform_batch_equals_single_solves_bitwise():
    name, dim, data, gold = [c for c in H.shipped_cases() if c[0] == "bar-72_input_0"][0]
    trusses = [Truss(dim).LoadFromJSON(data=data) for _ in range(5)]
    for k, t in enumerate(trusses):
        t.SetJointPosition(16 + (k % 4), tuple(v + 0.5 * k for v in t.GetJointPosition(16 + (k % 4))))
    SolveBatch(trusses)
    for t in trusses:
        s = Truss(dim).LoadFromJSON(data=t.Serialize())
        s.Solve()
        for k in H.FIELDS:
            assert np.array_equal(s._dense[k], t._dense[k]), k


def test_ga_fitness_vs_live_reference():
    g = H.load_json("live_ga_bar72.json")
    types = [MemberType(*row) for row in g["type_table"]]
    blocks = [(c, v, g["allow_stress"], g["allow_displace"]) for c, v in g["cases"].items()]
    blocks.append((g["tight"]["case"], g["tight"], g["tight"]["allow_stress"], g["tight"]["allow_displace"]))
    n_pen = 0
    for case, v, a_s, a_d in blocks:
        t = Truss(3).LoadFromJSON(f"{H.GOLDEN}/ref_data/{case}.json")
        for path in (0, 1, 2):
            t._get_plan().set_path(path)
            out = FitnessBatch(t, v["genes"], types, a_s, a_d)
            assert not out["info"].any()
            fit = np.array(v["fitness"])
            assert np.all(np.abs(out["fitness"] - fit) <= 1e-9 * np.abs(fit)), (case, path)
            assert out["flags"][:, 0].astype(bool).tolist() == v["stress_ok"]
            assert out["flags"][:, 1].astype(bool).tolist() == v["displace_ok"]
        n_pen += sum(1 for a, b in zip(v["stress_ok"], v["displace_ok"]) if not (a and b))
    assert n_pen > 0


def test_ga_class_uses_batched_fitness():
    import random
    from python_stable_3d_truss_analysis_b200.ga import GA
    g = H.load_json("live_ga_bar72.json")
    types = [MemberType(*row) for row in g["type_table"]]
    t = Truss(3).LoadFromJSON(f"{H.GOLDEN}/ref_data/bar-72_input_0.json")
    ga = GA(t, types, g["allow_stress"], g["allow_displace"], nIteration=3, nPop=64, nElite=16)
    v = g["cases"]["bar-72_input_0"]
    batch = ga.GetFitnessBatch(v["genes"][:8])
    for (f, s, d), fr, sr, dr in zip(batch, v["fitness"], v["stress_ok"], v["displace_ok"]):
        assert abs(f - fr) <= 1e-9 * abs(fr) and (s, d) == (sr, dr)
    single = ga.GetFitness(v["genes"][3])
    assert abs(single[0] - v["fitness"][3]) <= 1e-9 * abs(v["fitness"][3]) and t.isSolved
    random.seed(5)
    gene, info, pop, hist = ga.Evolve(isPrintMessage=False)
    assert len(pop) == 64 and len(hist) == 3 and hist == sorted(hist, reverse=True)


def test_load_cases_bar942_vs_live():
    z = np.load(f"{H.GOLDEN}/live_loadcases_bar942.npz")
    t = Truss(3).LoadFromJSON(f"{H.GOLDEN}/ref_data/bar-942_input_0.json")
    for path, independent in ((1, True), (2, True), (2, False)):   # (2, False): one factorisation, 16 substitutions
        t._get_plan().set_path(path)
        out = SolveLoadCases(t, z["F"], independent=independent)
        for b in range(z["F"].shape[0]):
            for k in H.FIELDS:
                err = orc.normwise_err(out[k][b], z[k][b])
                assert err <= H.TOL, (path, independent, b, k, err)


def test_member_type_batch_vs_oracle_bar942():
    rng = np.random.default_rng(3)
    data = json.load(open(f"{H.GOLDEN}/ref_data/bar-942_input_0.json"))
    joints, support, conn, aed, force = orc.arrays_from_json(data, 3)
    types = [MemberType(a, 1e4, 0.1) for a in (0.5, 1.0, 2.0, 4.0)]
    genes = rng.integers(0, 4, size=(3, conn.shape[0]))
    t = Truss(3).LoadFromJSON(data=data)
    tab = type_table(types)
    for path in (1, 2):
        t._get_plan().set_path(path)
        out = SolveMemberTypes(t, genes, types)
        for b in range(3):
            want = orc.solve_closed_form(3, joints, support, conn, tab[genes[b]], force)
            for k in H.FIELDS:
                assert orc.normwise_err(out[k][b], want[k]) <= H.TOL, (path, b, k)
            assert abs(out["weight"][b] - want["weight"]) <= 1e-9 * want["weight"]


def test_error_reporting_per_system():
    mt = MemberType(1, 1e7, 1)
    # counting rule (truss.py:158-164)
    u = Truss(3)
    for p, s in [((0, 0, 0), SupportType.PIN), ((1, 0, 0), SupportType.NO)]:
        u.AddNewJoint(p, s)
    u.AddNewMember(0, 1, mt)
    with pytest.raises(TrussNotStableError):
        u.Solve()
    # passes the counting rule but is a mechanism: a free joint hanging from one bar
    m = Truss(2)
    for p, s in [((0, 0), SupportType.PIN), ((4, 0), SupportType.PIN), ((2, 3), SupportType.NO), ((6, 3), SupportType.NO)]:
        m.AddNewJoint(p, s)
    for a, b in [(0, 2), (1, 2), (2, 3), (0, 1)]:
        m.AddNewMember(a, b, mt)
    m.AddExternalForce(3, (0, -1))
    assert m.isStable
    with pytest.raises(np.linalg.LinAlgError):
        m.Solve()
    assert not m.isSolved
    # zero-length member
    z = Truss(2)
    for p, s in [((0, 0), SupportType.PIN), ((4, 0), SupportType.PIN), ((2, 3), SupportType.NO), ((2, 3), SupportType.NO)]:
        z.AddNewJoint(p, s)
    for a, b in [(0, 2), (1, 2), (2, 3), (0, 3), (1, 3)]:
        z.AddNewMember(a, b, mt)
    with pytest.raises(ZeroDivisionError):
        z.Solve()
    # a batch reports per system and zero-fills the failures
    good = Truss(3).LoadFromJSON(f"{H.GOLDEN}/ref_data/bar-6_input_0.json")
    bad = Truss(3).LoadFromJSON(f"{H.GOLDEN}/ref_data/bar-6_input_0.json")
    bad.SetSupportType(0, SupportType.NO); bad.SetSupportType(1, SupportType.NO); bad.SetSupportType(3, SupportType.NO)
    info = SolveBatch([good, bad, good.Copy()], raise_on_error=False)
    assert info.tolist()[0] == 0 and info[1] != 0 and info[2] == 0
    assert good.isSolved and not bad.isSolved


def test_edge_cases():
    mt = MemberType(1, 1e7, 1)
    # every DOF supported: n = 0, reactions are zero, loads on supports are overwritten (truss.py:343,349)
    t = Truss(3)
    for p in [(0, 0, 0), (1, 0, 0), (0, 1, 0)]:
        t.AddNewJoint(p, SupportType.PIN)
    for a, b in [(0, 1), (1, 2), (0, 2)]:
        t.AddNewMember(a, b, mt)
    t.AddExternalForce(1, (5, 5, 5))
    t.Solve()
    assert t.GetDisplacements() == {} and t.GetExternalForces() == {} and t.GetInternalForces() == {}
    # no load at all: everything is zero
    name, dim, data, gold = H.shipped_cases()[0]
    data = dict(data); data["force"] = []
    t = Truss(dim).LoadFromJSON(data=data)
    t.Solve()
    assert not np.any(t._dense["u"]) and not np.any(t._dense["axial"])


def test_full_size_properties_bar942_x1024():
    """BASELINE configs[1] at full size: linearity in the load and bitwise determinism."""
    t = Truss(3).LoadFromJSON(f"{H.GOLDEN}/ref_data/bar-942_input_0.json")
    rng = np.random.default_rng(0)
    N = t.nJoint * 3
    base = rng.uniform(-10, 10, size=(4, N))
    coef = rng.uniform(-2, 2, size=(1024, 4))
    F = coef @ base
    out = SolveLoadCases(t, F, independent=True)
    again = SolveLoadCases(t, F, independent=True)
    for k in H.FIELDS:
        assert np.array_equal(out[k], again[k]), k                       # deterministic
    shared = SolveLoadCases(t, F)                                        # one factorisation, 1024 substitutions
    for k in H.FIELDS:
        assert orc.normwise_err(shared[k], out[k]) <= 2e-10, k     # (two different factorisation orders of a cond 6e6 matrix)
        assert np.array_equal(shared[k][100:140], SolveLoadCases(t, F[100:140])[k]), k   # batch-size independent
    basis = SolveLoadCases(t, base, independent=True)
    mask = t.GetDisplacementUnknownMask()
    for k in ("u", "axial"):
        want = coef @ basis[k]
        assert orc.normwise_err(out[k], want) <= 1e-9, k
    # equilibrium: reactions + applied loads on free DOFs sum to zero in every direction
    applied = np.where(mask, F, 0.0)
    react = np.where(~mask, out["ext"], 0.0)
    tot = (applied + react).reshape(1024, -1, 3).sum(axis=1)
    assert np.abs(tot).max() <= 1e-7 * np.abs(applied).sum(axis=1).max()


def test_ga_population_8192_properties():
    """BASELINE configs[2] at full size: batch == its own slices, and a sample against the oracle."""
    import random
    random.seed(0)
    types = [MemberType(i, random.uniform(1e7, 3e7), random.uniform(0.1, 1.0)) for i in range(1, 21)]
    genes = np.array([random.choices(range(20), k=72) for _ in range(8192)], dtype=np.int32)
    t = Truss(3).LoadFromJSON(f"{H.GOLDEN}/ref_data/bar-72_input_0.json")
    out = FitnessBatch(t, genes, types, 30000.0, 10.0)
    part = FitnessBatch(t, genes[4096:4160], types, 30000.0, 10.0)
    assert np.array_equal(out["fitness"][4096:4160], part["fitness"])
    data = json.load(open(f"{H.GOLDEN}/ref_data/bar-72_input_0.json"))
    joints, support, conn, _, force = orc.arrays_from_json(data, 3)
    tab = type_table(types)
    for b in (0, 777, 8191):
        f, s, d = orc.fitness(3, joints, support, conn, genes[b], tab, force, 30000.0, 10.0)
        assert abs(out["fitness"][b] - f) <= 1e-9 * abs(f) and tuple(out["flags"][b]) == (s, d)


def test_device_pointer_entry_point_matches_host_entry_point():
    import torch
    name, dim, data, gold = [c for c in H.shipped_cases() if c[0] == "bar-120_input_0"][0]
    t = Truss(dim).LoadFromJSON(data=data)
    xyz, support, conn, aed, force = t._pack()
    plan = t._get_plan()
    B = 7
    host = plan.solve_host(B, xyz, force, aed=aed)
    dev = torch.device("cuda:0")
    td = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    out = {"u": torch.empty(B, plan.N, dtype=torch.float64, device=dev), "ext": torch.empty(B, plan.N, dtype=torch.float64, device=dev),
           "axial": torch.empty(B, plan.M, dtype=torch.float64, device=dev), "weight": torch.empty(B, dtype=torch.float64, device=dev),
           "info": torch.empty(B, dtype=torch.int32, device=dev)}
    plan.solve_device(B, td(xyz), td(force), aed=td(aed), out=out)
    torch.cuda.synchronize()
    for k in ("u", "ext", "axial", "weight"):
        assert np.array_equal(out[k].cpu().numpy(), host[k]), k
    H.assert_close({k: host[k][0] for k in H.FIELDS} | {"weight": host["weight"][0]}, gold, what=name)


def test_fp64_peaks_are_measurable():
    for which in (0, 1):
        tf, ms = _lib.fp64_peak(which, 1024)
        assert tf > 1.0 and ms > 0


def test_config4_ragged_65536_properties():
    """BASELINE configs[3] at full size: 65536 ragged cube-7 systems (pool tiled with joint jitter) in one call:
    a sample against the oracle, determinism, and equality with the same systems solved in a smaller batch."""
    pool = [Truss(3).LoadFromJSON(data={k: g[k] for k in ("joint", "force", "member")}) for g in H.load_json("live_cube7_aug.json")]
    B = 65536
    jo, mo, xyz, sup, conn, aed, force, which = H.ragged_pool_arrays(pool, B)
    out = _lib.solve_ragged_host(3, jo, mo, xyz, sup, conn, aed, force)
    assert not out["info"].any()
    again = _lib.solve_ragged_host(3, jo, mo, xyz, sup, conn, aed, force)
    for k in H.FIELDS:
        assert np.array_equal(out[k], again[k]), k
    # a slice of the batch solved on its own gives the same bits
    lo, hi = 40000, 40064
    sub = _lib.solve_ragged_host(3, jo[lo:hi + 1] - jo[lo], mo[lo:hi + 1] - mo[lo], xyz[jo[lo] * 3:jo[hi] * 3], sup[jo[lo]:jo[hi]],
                                 conn[mo[lo] * 2:mo[hi] * 2], aed[mo[lo] * 3:mo[hi] * 3], force[jo[lo] * 3:jo[hi] * 3])
    assert np.array_equal(sub["u"], out["u"][jo[lo] * 3:jo[hi] * 3]) and np.array_equal(sub["axial"], out["axial"][mo[lo]:mo[hi]])
    for b in (0, 1, 12345, 65535):
        j0, j1, m0, m1 = jo[b], jo[b + 1], mo[b], mo[b + 1]
        want = orc.solve(3, xyz[j0 * 3:j1 * 3].reshape(-1, 3), sup[j0:j1], conn[m0 * 2:m1 * 2].reshape(-1, 2),
                         aed[m0 * 3:m1 * 3].reshape(-1, 3), force[j0 * 3:j1 * 3])
        got = {"u": out["u"][j0 * 3:j1 * 3], "ext": out["ext"][j0 * 3:j1 * 3], "axial": out["axial"][m0:m1], "weight": out["weight"][b]}
        H.assert_close(got, want, what=f"config4[{b}]")


def test_config5_cube12_tiled_vs_oracle():
    """BASELINE configs[4] shape (12^3 cube truss: nJ 2197, M 14868, n 6084) through the tiled pipeline, two systems with
    different member areas, against the oracle's dense solve; equilibrium of loads and reactions."""
    t = H.cube_truss(12)
    xyz, support, conn, aed, force = t._pack()
    plan = t._get_plan()
    assert plan.n == 6084 and plan.path == 1
    rng = np.random.default_rng(5)
    B = 2
    aedb = np.repeat(aed[None], B, axis=0).copy()
    aedb[:, :, 0] = rng.uniform(1.0, 20.0, size=(B, plan.M))
    out = plan.solve_host(B, xyz, force, aed=aedb)
    assert not out["info"].any()
    mask = np.asarray(t.GetDisplacementUnknownMask())
    for b in range(B):
        want = orc.solve_closed_form(3, xyz, support, conn, aedb[b], force)
        H.assert_close({k: out[k][b] for k in H.FIELDS} | {"weight": out["weight"][b]}, want, what=f"cube12[{b}]")
        tot = (np.where(mask, force, 0.0) + np.where(~mask, out["ext"][b], 0.0)).reshape(-1, 3).sum(axis=0)
        assert np.abs(tot).max() <= 1e-7 * np.abs(force).sum()


def test_band_kernels_agree_bitwise_across_batch_sizes(tmp_path):
    """A system's band-path result does not depend on the batch it is in (SURVEY.md section 4 (iv): bit-identical per
    truss across GPU counts / shard sizes).  k_band_ts: 4096 systems (seven CTAs per SM, several systems per CTA in the
    grid-stride loop) against 32 of them (one system per CTA).  The 16x16 kernels (TB_BAND_LEGACY=1, a fresh process):
    the two-warp k_band2 at 4096 systems against the three-warp k_band3 at 32, same arithmetic in the same order."""
    e = BC.get("bar-942")
    plan = BC.plan_for(e)
    NB16, nb = plan.info.band_blocks, BC.ts_nb(plan.ts_program())
    xyz, aed, F = BC.inputs(plan, e, 4096, seed=3)
    big, seen_big = H.cuda_kernels(lambda: H.solve_device_np(plan, 4096, xyz, aed, F))
    small, seen_small = H.cuda_kernels(lambda: H.solve_device_np(plan, 32, xyz, aed[1000:1032], F[1000:1032]))
    print(f"k_band_ts: {seen_big} | {seen_small}")
    assert H.band_kernels(seen_big) == H.band_kernels(seen_small) == [f"k_band_ts<{nb}>"], (seen_big, seen_small)
    for k in ("u", "ext", "axial", "weight", "info"):
        assert np.array_equal(big[k][1000:1032], small[k]), k
    (lbig, lseen_big), (lsmall, lseen_small) = H.run_band_child(tmp_path, {"TB_BAND_LEGACY": "1"}, [
        {"label": "bar-942", "B": 4096, "seed": 3}, {"label": "bar-942", "B": 4096, "seed": 3, "slice": [1000, 1032]}])
    print(f"legacy: {lseen_big} | {lseen_small}")
    assert H.band_kernels(lseen_big) == [f"k_band2<{NB16}>"] and H.band_kernels(lseen_small) == [f"k_band3<{NB16}>"]
    for k in ("u", "ext", "axial", "weight", "info"):
        assert np.array_equal(lbig[k][1000:1032], lsmall[k]), k
    assert not big["info"].any() and not lbig["info"].any()
    joints, support, conn, _, _ = BC.arrays(e)
    for b in (0, 1000, 4095):
        want = orc.solve(3, joints, support, conn, aed[b], F[b])
        for name, got in (("k_band_ts", big), ("k_band2", lbig)):
            H.assert_close({k: got[k][b] for k in H.FIELDS} | {"weight": got["weight"][b]}, want, what=f"{name}[{b}]")


def test_band_kernel_variants_agree_bitwise(tmp_path):
    """k_band1 (one warp per system), k_band2 (two) and k_band3 (three) are the same arithmetic in the same order.
    Under TB_BAND_LEGACY=1 (systems with a two-sided program take the 16x16 kernels too) each is forced in turn through
    TB_BAND_WARPS (both are read once per process, hence the subprocesses) on the band catalogue's systems of
    NB16 = 1 .. 5: they return the same bits, and each matches the oracle.  NB16 = 6 .. 8 run on k_band1 alone, at 5
    systems: not a multiple of its systems per CTA (4 for NB16 <= 6, 2 for 7 and 8)."""
    systems = [e for e in BC.catalogue() if "/" not in e.label]
    NB16 = {e.label: BC.plan_for(e).info.band_blocks for e in systems}
    narrow = [e.label for e in systems if NB16[e.label] <= 5]
    assert sorted({NB16[x] for x in narrow}) == [1, 2, 3, 4, 5]
    assert sorted({v for v in NB16.values() if v > 5}) == [6, 7, 8]
    B = 5
    res = {}
    for w in (1, 2, 3):
        labels = [e.label for e in systems] if w == 1 else narrow
        runs = H.run_band_child(tmp_path, {"TB_BAND_LEGACY": "1", "TB_BAND_WARPS": str(w)},
                                [{"label": x, "B": B, "seed": 11} for x in labels])
        for x, (out, seen) in zip(labels, runs):
            print(f"TB_BAND_WARPS={w} {x}: {seen}")
            assert H.band_kernels(seen) == [f"k_band{w}<{NB16[x]}>"], (w, x, seen)
            assert not out["info"].any(), (w, x)
            res[w, x] = out
    for x in narrow:
        for w in (2, 3):
            for k in ("u", "ext", "axial", "weight"):
                assert np.array_equal(res[1, x][k], res[w, x][k]), (x, w, k)
    for e in systems:
        plan = BC.plan_for(e)
        joints, support, conn, _, _ = BC.arrays(e)
        xyz, aed, F = BC.inputs(plan, e, B, seed=11)
        for b in range(B):
            want = orc.solve(e.dim, joints, support, conn, aed[b], F[b])
            got = res[1, e.label]
            H.assert_close({k: got[k][b] for k in H.FIELDS} | {"weight": got["weight"][b]}, want, what=f"k_band1 {e.label}[{b}]")
            be = H.backward_error(e.dim, joints, support, conn, aed[b], F[b], got["u"][b])
            assert be <= 1e-14, (e.label, b, be)


def test_pivot_rsqrt_accuracy():
    """The 16x16 pivot blocks take 1/sqrt(pivot) from the hardware seed plus one third-order correction
    (tb_blocks.cuh: rsqrt_pos); it must stay within 2 ulp of 1/sqrt(d) over the whole accepted pivot range."""
    from python_stable_3d_truss_analysis_b200 import _lib
    assert _lib.rsqrt_probe(1 << 22) <= 4.5e-16


@pytest.mark.parametrize("dim,per_level,levels", [(2, 2, 40), (3, 3, 30), (3, 5, 24), (3, 8, 16), (3, 11, 12), (3, 13, 10),
                                                   (3, 15, 9), (3, 19, 8), (3, 21, 7)])
def test_band_path_every_band_width_vs_oracle(dim, per_level, levels):
    """Towers of growing cross-section sweep the number of sub-diagonal 16x16 blocks of the band path (1 .. 8: the
    three-warp / two-warp kernels up to 5, the one-warp kernel beyond), each against the oracle, with a factorisation
    per load case and with the shared one."""
    data = _tower(dim, per_level, levels, seed=per_level)
    t = Truss(dim).LoadFromJSON(data=data)
    plan = t._get_plan()
    if plan.info.band_blocks > 8:
        pytest.skip(f"band of {plan.info.band_blocks} blocks: not a band-path system")
    plan.set_path(2)
    joints, support, conn, aed, force = orc.arrays_from_json(data, dim)
    rng = np.random.default_rng(1)
    F = np.stack([force, -0.5 * force, force * rng.uniform(0.5, 2.0, size=force.shape)])
    for independent in (True, False):
        out = SolveLoadCases(t, F, independent=independent)
        for b in range(3):
            want = orc.solve(dim, joints, support, conn, aed, F[b])
            for k in H.FIELDS:
                err = orc.normwise_err(out[k][b], want[k])
                assert err <= H.TOL, (plan.info.band_blocks, independent, b, k, err)


@pytest.mark.parametrize("dim,per_level,levels,path", [(2, 4, 40, 2), (2, 9, 30, 2), (2, 9, 30, 1), (3, 8, 16, 1), (3, 13, 10, 1)])
def test_towers_2d_and_tiled_path_vs_oracle(dim, per_level, levels, path):
    """2D band systems and the same kind of tower through the tiled (64x64 block-sparse) pipeline."""
    data = _tower(dim, per_level, levels, seed=100 + per_level)
    t = Truss(dim).LoadFromJSON(data=data)
    t._get_plan().set_path(path)
    t.Solve()
    want = orc.solve(dim, *orc.arrays_from_json(data, dim))
    for k in H.FIELDS:
        err = orc.normwise_err(t._dense[k], want[k])
        assert err <= H.TOL, (path, k, err)


def test_long_tower_shared_factor_falls_back_to_warp_per_load_case():
    """A band system too long for y to stay in shared memory (196 block columns): tb_solve_loadcases uses the
    warp-per-load-case substitution kernel instead of the tensor-core tile kernel.  The tower (pinned at both ends, loaded
    at mid-height) is slender: cond(K_ff) = 1.8e8, where the reference's LU and a Cholesky factorisation on the CPU already
    differ by ~1e-9, so this test checks the kernels at 1e-7 instead of the 1e-9 of the well-conditioned fixtures."""
    data = _tower(3, 3, 350, seed=7)
    for j in data["joint"][-3:]:
        j[1] = "PIN"
    rng = np.random.default_rng(9)
    data["force"] = [[3 * lv + k, [float(x) for x in rng.uniform(-5, 5, size=3)]] for lv in (120, 175, 230) for k in range(3)]
    t = Truss(3).LoadFromJSON(data=data)
    plan = t._get_plan()
    assert plan.info.path == 2 and plan.info.n_free > 3040
    joints, support, conn, aed, force = orc.arrays_from_json(data, 3)
    F = np.stack([force, 2.0 * force, -force, 0.25 * force, force[::-1].copy()])
    shared = SolveLoadCases(t, F)
    indep = SolveLoadCases(t, F, independent=True)
    for b in (0, 4):
        want = orc.solve(3, joints, support, conn, aed, F[b])
        for k in H.FIELDS:
            assert orc.normwise_err(shared[k][b], want[k]) <= 1e-7, ("shared", b, k)
            assert orc.normwise_err(indep[k][b], want[k]) <= 1e-7, ("independent", b, k)


@pytest.mark.parametrize("path", [1, 2], ids=["tiled", "band"])
def test_blocked_paths_report_failures_per_system(path):
    """A system whose stiffness matrix is not positive definite (all members of zero stiffness) fails alone: info > 0
    (first non-positive pivot, 1-based) and zero-filled outputs for it, correct results for its batch mates; with the
    factorisation shared, the failure reaches every load case."""
    data = _tower(3, 5, 24, seed=3)
    t = Truss(3).LoadFromJSON(data=data)
    t._get_plan().set_path(path)
    types = [MemberType(1.0, 1e4, 0.1), MemberType(1.0, 0.0, 0.1)]
    genes = np.zeros((3, t.nMember), dtype=np.int32)
    genes[1, :] = 1
    out = SolveMemberTypes(t, genes, types, raise_on_error=False)
    assert out["info"][0] == 0 and out["info"][2] == 0 and out["info"][1] > 0
    assert not np.any(out["u"][1]) and not np.any(out["axial"][1]) and not np.any(out["ext"][1])
    assert np.array_equal(out["u"][0], out["u"][2]) and np.any(out["u"][0])
    with pytest.raises(np.linalg.LinAlgError):
        SolveMemberTypes(t, genes, types)
    for m in range(t.nMember):                 # the truss itself with zero stiffness: every load case fails
        t.SetMemberType(m, types[1])
    N = t.nJoint * 3
    res = SolveLoadCases(t, np.ones((4, N)), raise_on_error=False)
    assert np.all(res["info"] > 0) and not np.any(res["u"])


def _k_reference_with_device_squares(dim, joints, conn, aed, row, col, ptr, mem, loc):
    """GetKMatrix()[mask][:, mask] entries (truss.py:307-316, 343) with the squares of the cosines taken as products: the
    reference's ``l ** 2.`` goes through libm pow, which is an ulp off the product now and then (no GPU reproduces libm)."""
    from tests import ts_replay
    prods = [ts_replay.member_products(dim, joints, conn[m], aed[m][0], aed[m][1]) for m in range(conn.shape[0])]
    out = np.zeros(len(row))
    for i in range(len(row)):
        v = 0.0
        for q in range(ptr[i], ptr[i + 1]):
            a, b = divmod(int(loc[q]), 2 * dim)
            k, c = prods[mem[q]]
            t = k * (c[a % dim] * c[b % dim])
            v = v + (-t if (a // dim) != (b // dim) else t)
        out[i] = v
    return out


@pytest.mark.parametrize("name,dim,data,gold", [c for c in H.shipped_cases() if c[0].split("_")[0] in ("bar-6", "bar-10", "bar-72", "bar-942")],
                         ids=lambda v: v if isinstance(v, str) else None)
def test_device_assembled_K_is_bit_exact(name, dim, data, gold):
    """SURVEY section 7 step-2 gate: the K_ff values the DEVICE assembles (its own roundings of length, EA/L, cosines, the
    products and the ascending-member sums) equal the reference's reduced stiffness matrix bit for bit."""
    joints, support, conn, aed, force = orc.arrays_from_json(data, dim)
    for path in (2, 1):
        plan = _lib.Plan(dim, conn, support)
        try:
            plan.set_path(path)
        except _lib.TrussLibError:
            continue
        kv = plan.assemble_host(2, joints, aed)
        row, col, ptr, mem, loc = plan.scatter()
        want = _k_reference_with_device_squares(dim, joints, conn, aed, row, col, ptr, mem, loc)
        assert np.array_equal(kv[0], want) and np.array_equal(kv[1], want), (name, path)
        K = orc.assemble_K(dim, joints, conn, aed)
        mask = orc.free_mask(dim, support)
        ref = K[mask][:, mask][row, col]
        mism = np.count_nonzero(kv[0] != ref)
        # the oracle itself (CPython's compensated sum() in the length, pow for the squares) may sit an ulp away
        assert mism <= 0.02 * len(ref) + 2 and np.all(np.abs(kv[0] - ref) <= 1e-12 * np.abs(ref).max()), (name, path, mism)


def test_two_streams_and_two_threads_share_one_plan():
    """ADVICE r1: a plan owns one workspace; calls from two streams / two threads must serialise, not corrupt each other."""
    import threading
    import torch
    name, dim, data, gold = next(c for c in H.shipped_cases() if c[0].startswith("bar-942"))
    t = Truss(dim).LoadFromJSON(data=data)
    xyz, sup, conn, aed, force = t._pack()
    plan = t._get_plan()
    dev = torch.device("cuda:0")
    td = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    B = 64
    rng = np.random.default_rng(7)
    Fs = [rng.uniform(-10, 10, size=(B, plan.N)) for _ in range(2)]
    dx, da = td(xyz), td(aed)
    dF = [td(F) for F in Fs]
    outs = [{k: torch.empty(B, plan.N if k in ("u", "ext") else plan.M, dtype=torch.float64, device=dev) for k in ("u", "ext", "axial")}
            for _ in range(2)]
    for o in outs:
        o["weight"] = torch.empty(B, dtype=torch.float64, device=dev)
        o["info"] = torch.empty(B, dtype=torch.int32, device=dev)
    ref = [plan.solve_host(B, xyz, F, aed=aed) for F in Fs]
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]

    def work(i):
        for _ in range(20):
            plan.solve_device(B, dx, dF[i], aed=da, out=outs[i], stream=streams[i])

    th = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for x in th:
        x.start()
    for x in th:
        x.join()
    torch.cuda.synchronize()
    for i in range(2):
        for k in ("u", "ext", "axial"):
            assert np.array_equal(outs[i][k].cpu().numpy(), ref[i][k]), (i, k)


def test_one_process_two_devices():
    """VERDICT r1 #8: kernel attributes / helper streams are per device; a plan refuses to run on a device it was not made on."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    name, dim, data, gold = next(c for c in H.shipped_cases() if c[0].startswith("bar-942"))
    res = []
    for d in (0, 1):
        torch.cuda.set_device(d)
        t = Truss(dim).LoadFromJSON(data=data)
        t.Solve()
        H.assert_close(dense(t), gold, what=f"device {d}")
        res.append(t._dense["u"].copy())
        if d == 1:
            plan1 = t._get_plan()
    assert np.array_equal(res[0], res[1])
    torch.cuda.set_device(0)
    xyz, sup, conn, aed, force = t._pack()
    with pytest.raises(_lib.TrussLibError) as ei:
        plan1.solve_host(1, xyz, force, aed=aed)
    assert ei.value.code == -9
    torch.cuda.set_device(0)


@pytest.mark.gpu
def test_pipelined_host_calls_match_blocking_calls():
    """tb_solve_host_async / tb_host_wait: five batches streamed with two in flight give the bits of tb_solve_host,
    tickets complete in order, a blocking call in between drains the pipeline, and a bad ticket is refused."""
    name, dim, data, _ = next(c for c in H.shipped_cases() if c[0].startswith("bar-942"))
    t = Truss(dim).LoadFromJSON(data=data)
    xyz, sup, conn, aed, force = t._pack()
    plan = t._get_plan()
    rng = np.random.default_rng(5)
    B = 37
    Fs = [rng.uniform(-10, 10, size=(B, plan.N)) for _ in range(5)]
    want = [plan.solve_host(B, xyz, F, aed=aed) for F in Fs]
    pinned = []
    for F in Fs:
        h = _lib.pinned_empty(F.shape)
        h[...] = F
        pinned.append(h)
    outs, tickets = [], []
    for i, F in enumerate(pinned):
        tk, out = plan.solve_host_async(B, xyz, F, aed=aed)
        tickets.append(tk)
        outs.append(out)
        if i >= 1:
            plan.host_wait(tickets[i - 1])
            for k in ("u", "ext", "axial", "weight"):
                assert np.array_equal(outs[i - 1][k], want[i - 1][k]), (i - 1, k)
    assert tickets == sorted(tickets) and len(set(tickets)) == len(tickets)
    again = plan.solve_host(B, xyz, Fs[0], aed=aed)          # a blocking call first waits for everything in flight
    for k in ("u", "ext", "axial", "weight"):
        assert np.array_equal(outs[-1][k], want[-1][k]), k
        assert np.array_equal(again[k], want[0][k]), k
    plan.host_wait(tickets[-1])                               # already complete: returns at once
    with pytest.raises(_lib.TrussLibError):
        plan.host_wait(tickets[-1] + 7)


@pytest.mark.gpu
def test_fixed_member_type_double_solve_matches_oracle():
    """SolveWithFixedMemberType (data.py:17-44, 108-114): every truss solved as it is and again with all members of the
    fixed type, in two batched calls -- against the oracle run on arrays with the member properties replaced, on a
    ragged list (cube-7 trusses) and on a uniform one (copies of bar-72 with different member types)."""
    from python_stable_3d_truss_analysis_b200.batch import SolveWithFixedMemberType

    fixed = MemberType(1., 1e7, 0.1)
    ragged = [Truss(d).LoadFromJSON(data=data) for _, d, data, _ in H.cube7_shipped()[:6]]
    name, dim, data, _ = next(c for c in H.shipped_cases() if c[0].startswith("bar-72"))
    uniform = []
    for i in range(4):
        t = Truss(dim).LoadFromJSON(data=data)
        for m in t.GetMemberIDs():
            t.SetMemberType(m, MemberType(1.0 + 0.25 * ((m + i) % 5), 1e7, 0.1))
        uniform.append(t)
    for trusses in (ragged, uniform):
        res = SolveWithFixedMemberType(trusses, fixed)
        den = SolveWithFixedMemberType(trusses, fixed, dense=True)
        assert len(res) == len(trusses)
        for i, t in enumerate(trusses):
            assert t.isSolved
            xyz, sup, conn, aed, force = t._pack()
            own = orc.solve(t.dim, xyz, sup, conn, aed, force.reshape(-1, t.dim))
            assert orc.normwise_err(t._dense["u"], own["u"]) <= 1e-9
            aed2 = np.tile(np.array(fixed.Serialize()), (conn.shape[0], 1))
            want = orc.solve(t.dim, xyz, sup, conn, aed2, force.reshape(-1, t.dim))
            assert orc.normwise_err(den["u"][i], want["u"]) <= 1e-9
            assert orc.normwise_err(den["stress"][i], want["axial"] / fixed.a) <= 1e-9
            internals, displaces = res[i]
            for m, s in internals.items():
                assert abs(s - want["axial"][m] / fixed.a) <= 1e-9 * np.abs(want["axial"]).max() / fixed.a
            big = np.nonzero(np.abs(want["axial"]) > 1e-8)[0]
            assert set(big.tolist()) <= set(internals)
            wu = want["u"].reshape(-1, t.dim)
            for j, v in displaces.items():
                assert np.abs(v - wu[j]).max() <= 1e-9 * np.abs(wu).max()


@pytest.mark.gpu
@pytest.mark.parametrize("case,path", [("bar-72", 0), ("bar-72", 1), ("bar-942", 2), ("bar-942", 1), ("bar-10", 0)])
def test_compact_outputs_equal_the_dense_ones(case, path):
    """tb_batch_out.u_free / react (the compact layout: n + s + M doubles per system) against the dense outputs, bit for
    bit, on every pipeline and through the device, blocking-host and pipelined-host entry points, with and without the
    dense arrays in the same call; expanding them gives back u and ext (truss.py:342-351)."""
    import torch
    name, dim, data, _ = next(c for c in H.shipped_cases() if c[0].startswith(case))
    t = Truss(dim).LoadFromJSON(data=data)
    xyz, sup, conn, aed, force = t._pack()
    plan = _lib.Plan(dim, conn, sup.astype(np.uint8))
    plan.set_path(path)
    free_idx, _, sup_idx = plan.maps()
    B = 19
    rng = np.random.default_rng(11)
    F = force.reshape(1, -1) * rng.uniform(0.5, 2.0, size=(B, 1)) + rng.uniform(-1, 1, size=(B, plan.N))
    dense = plan.solve_host(B, xyz, F, aed=aed)
    assert not dense["info"].any()
    want_u, want_r = dense["u"][:, free_idx], dense["ext"][:, sup_idx]
    # blocking host call: compact only, and compact next to dense
    only = plan.solve_host(B, xyz, F, aed=aed, want=("u_free", "react", "axial", "weight"))
    both = plan.solve_host(B, xyz, F, aed=aed, want=("u", "ext", "u_free", "react", "axial"))
    for got in (only, both):
        assert np.array_equal(got["u_free"], want_u) and np.array_equal(got["react"], want_r)
        assert np.array_equal(got["axial"], dense["axial"])
    assert np.array_equal(both["u"], dense["u"]) and np.array_equal(both["ext"], dense["ext"])
    u, ext = plan.expand_compact(only["u_free"], only["react"], F)
    assert np.array_equal(u, dense["u"]) and np.array_equal(ext, dense["ext"])
    # pipelined host call
    Fp = _lib.pinned_empty(F.shape)
    Fp[...] = F
    tk, pout = plan.solve_host_async(B, xyz, Fp, aed=aed, want=("u_free", "react", "axial"))
    plan.host_wait(tk)
    assert np.array_equal(pout["u_free"], want_u) and np.array_equal(pout["react"], want_r)
    # device entry point
    dev = torch.device("cuda:0")
    td = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)   # noqa: E731
    dout = {"u_free": torch.empty(B, plan.n, dtype=torch.float64, device=dev), "react": torch.empty(B, plan.s, dtype=torch.float64, device=dev),
            "axial": torch.empty(B, plan.M, dtype=torch.float64, device=dev), "info": torch.empty(B, dtype=torch.int32, device=dev)}
    plan.solve_device(B, td(xyz), td(F), aed=td(aed), out=dout)
    torch.cuda.synchronize()
    assert np.array_equal(dout["u_free"].cpu().numpy(), want_u) and np.array_equal(dout["react"].cpu().numpy(), want_r)
    # ragged batches have no common n / s: the compact layout is refused there
    jo, mo = np.array([0, xyz.shape[0]], np.int64), np.array([0, conn.shape[0]], np.int64)
    ri = _lib.TbRaggedIn(dim, 1, jo.ctypes.data, mo.ctypes.data, xyz.ctypes.data, sup.astype(np.uint8).ctypes.data, conn.ctypes.data,
                         aed.ctypes.data, force.ctypes.data, xyz.shape[0], conn.shape[0])
    bo = _lib.TbBatchOut(None, None, None, None, None, only["u_free"].ctypes.data, None)
    assert _lib.lib().tb_solve_ragged_host(C.byref(ri), C.byref(bo)) == -3


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["bar-72", "bar-25", "bar-120", "bar-10", "bar-47"])
def test_uniform_and_ragged_entry_points_agree_bitwise(case):
    """The same trusses through the plan's uniform batch (tb_solve_host) and as a ragged batch (tb_solve_ragged_host):
    the warp-per-truss kernel sums every K entry in ascending member order either way (truss.py:307-316) -> the same bits."""
    name, dim, data, _ = next(c for c in H.shipped_cases() if c[0].startswith(case))
    t = Truss(dim).LoadFromJSON(data=data)
    xyz, sup, conn, aed, force = t._pack()
    plan = _lib.Plan(dim, conn, sup.astype(np.uint8))
    if plan.info.path != 0:
        pytest.skip("not a small-path truss")
    B = 5
    rng = np.random.default_rng(2)
    xyzb = xyz[None] + rng.normal(0, 0.01, size=(B,) + xyz.shape)
    aedb = aed[None] * rng.uniform(0.5, 2.0, size=(B, aed.shape[0], 1))
    F = force.reshape(1, -1) * rng.uniform(0.5, 2.0, size=(B, 1))
    uni = plan.solve_host(B, xyzb, F, aed=aedb)
    nJ, M = xyz.shape[0], conn.shape[0]
    jo, mo = np.arange(B + 1, dtype=np.int64) * nJ, np.arange(B + 1, dtype=np.int64) * M
    rag = _lib.solve_ragged_host(dim, jo, mo, xyzb.reshape(-1), np.tile(sup.astype(np.uint8), B), np.tile(conn.reshape(-1), B),
                                 aedb.reshape(-1), F.reshape(-1))
    assert not uni["info"].any() and not rag["info"].any()
    # (a ragged batch sizes shared memory for d * nJ free DOFs; bar-120 then no longer fits the warp kernel and runs on the
    # CTA-per-truss kernel, another summation order: equal to rounding there, bit for bit everywhere else)
    same_kernel = _lib.lib().tb_small_path_fits(dim, nJ, M) and case != "bar-120"
    for k in ("u", "ext", "axial", "weight"):
        a_, b_ = np.asarray(uni[k]).reshape(-1), np.asarray(rag[k]).reshape(-1)
        if same_kernel:
            assert np.array_equal(a_, b_), k
        else:
            assert orc.normwise_err(a_, b_) <= 1e-9, k


@pytest.mark.gpu
def test_shared_divisor_division_is_ieee_division():
    """The member geometry divides EA and the three coordinate differences by the member length (truss.py:19, 56-63) with
    one correctly rounded reciprocal and Markstein's multiply / FMA / FMA per numerator: bit for bit the quotients of IEEE
    division on 300 M operand pairs, random and adversarial (significands of all ones, powers of two, extreme exponents)."""
    for seed in (1, 2, 3):
        m = C.c_uint64(1)
        _lib.check(_lib.lib().tb_div_probe(100_000_000, seed, C.byref(m)))
        assert m.value == 0, (seed, m.value)
