"""Ragged batches beyond the fused kernels on the GPU: the envelope kernel k_rag_env (tb_solve_ragged_env,
tb_ragged_env_order) and the routing of tb_solve_ragged.  Oracle parity (1e-9 norm-wise per field), the ordering hook
against the plan's rule, routing and bit identity, determinism and batch independence, failure classes among good
trusses, the host entry point, and the scratch arena across streams and CUDA graphs."""
import json

import numpy as np
import pytest

from oracle import truss_oracle as orc
from python_stable_3d_truss_analysis_b200 import _lib
from tests import helpers as H
from tests import ragged_order as RO

pytestmark = pytest.mark.gpu

FIELDS = ("u", "ext", "axial", "weight")


def _torch():
    import torch
    return torch


def fixtures(dim):
    """(name, (joints, support, conn, aed, force)) of every shipped fixture of this dim and every live_random entry."""
    out = []
    for name, d, data, _ in H.shipped_cases():
        if d == dim and "_input_" in name:
            out.append((name, tuple(orc.arrays_from_json(data, dim))))
    for i, c in enumerate(H.load_json("live_random.json")):
        if c["dim"] == dim:
            out.append((f"random{i}", tuple(orc.arrays_from_json(c["data"], dim))))
    return out


def cube7_aug():
    return [(f"aug{i}", tuple(orc.arrays_from_json(d, 3))) for i, d in enumerate(H.load_json("live_cube7_aug.json"))]


def pack(trusses):
    nj = [len(t[0]) for t in trusses]
    nm = [len(t[2]) for t in trusses]
    jo, mo = np.zeros(len(trusses) + 1, np.int64), np.zeros(len(trusses) + 1, np.int64)
    jo[1:], mo[1:] = np.cumsum(nj), np.cumsum(nm)
    cat = lambda i, dt: np.concatenate([np.asarray(t[i], dt).reshape(-1) for t in trusses])  # noqa: E731
    return {"joint_off": jo, "member_off": mo, "xyz": cat(0, np.float64), "support": cat(1, np.uint8),
            "conn": cat(2, np.int32), "aed": cat(3, np.float64), "force": cat(4, np.float64)}


def unpack(p, dim, b):
    """(joints, support, conn, aed, force) of truss b of a packed numpy batch."""
    j0, j1, m0, m1 = (int(x) for x in (p["joint_off"][b], p["joint_off"][b + 1], p["member_off"][b], p["member_off"][b + 1]))
    return (p["xyz"][j0 * dim:j1 * dim].reshape(-1, dim), p["support"][j0:j1], p["conn"][2 * m0:2 * m1].reshape(-1, 2),
            p["aed"][3 * m0:3 * m1].reshape(-1, 3), p["force"][j0 * dim:j1 * dim])


def rows(res, p, dim, b):
    j0, j1, m0, m1 = (int(x) for x in (p["joint_off"][b], p["joint_off"][b + 1], p["member_off"][b], p["member_off"][b + 1]))
    return {"u": res["u"][j0 * dim:j1 * dim], "ext": res["ext"][j0 * dim:j1 * dim], "axial": res["axial"][m0:m1],
            "weight": res["weight"][b:b + 1], "info": res["info"][b:b + 1]}


def to_dev(p):
    torch = _torch()
    return {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in p.items() if isinstance(v, np.ndarray)}


def run(fn, dim, p, **kw):
    """fn (solve_ragged_device / solve_ragged_env_device) on a packed numpy batch under torch.profiler: numpy results and
    the names of the kernels that ran."""
    torch = _torch()
    from torch.profiler import ProfilerActivity, profile

    d = to_dev(p)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn(dim, d, **kw)
        torch.cuda.synchronize()
    names = {ev.name for ev in prof.events()}
    return {k: v.cpu().numpy() for k, v in out.items()}, names


def ran(names, kernel):
    return any(kernel in n for n in names)


def check_oracle(res, p, dim, names=None):
    B = len(p["joint_off"]) - 1
    idx = range(B) if names is None else names
    failed = [(b, int(res["info"][b])) for b in idx if res["info"][b] != 0]
    assert not failed, failed
    for b in idx:
        t = unpack(p, dim, b)
        want = orc.solve(dim, *t)
        got = rows(res, p, dim, b)
        for k in FIELDS:
            err = orc.normwise_err(np.atleast_1d(got[k]), np.atleast_1d(want[k]))
            assert err <= 1e-9, (b, k, err)


@pytest.mark.parametrize("dim", [2, 3])
def test_env_kernel_matches_oracle_on_fixtures(dim):
    cases = fixtures(dim) + (cube7_aug() if dim == 3 else [])
    p = pack([t for _, t in cases])
    res, names = run(_lib.solve_ragged_env_device, dim, p)
    assert ran(names, "k_rag_env"), names
    assert not ran(names, "k_dense16") and not ran(names, "k_small")
    check_oracle(res, p, dim)
    if dim == 3:
        assert any(n.startswith("bar-942") for n, _ in cases)                 # 732 DOFs


def _generated(num_cube, n, seed):
    from python_stable_3d_truss_analysis_b200.generate import GenerateRandomCubeTrussesOnDevice

    return GenerateRandomCubeTrussesOnDevice(n, gridRange=(6, 6, 6), numCubeRange=(num_cube, num_cube),
                                            lengthRange=(100, 200), isDoStructuralAnalysis=True, seed=seed)


@pytest.mark.parametrize("num_cube,n", [(20, 256), (40, 256), (80, 64), (216, 8)])
def test_generated_large_trusses_solve_through_tb_solve_ragged(num_cube, n):
    torch = _torch()
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        g = _generated(num_cube, n, seed=num_cube)
        torch.cuda.synchronize()
    assert ran({ev.name for ev in prof.events()}, "k_rag_env")
    assert (g["gen_info"] == 0).all()
    assert (g["info"] == 0).all(), np.unique(g["info"], return_counts=True)
    nj = np.diff(g["joint_off"])
    sample = sorted({int(np.argmax(nj)), int(np.argmin(nj)), 0, n - 1})
    check_oracle(g, g, 3, names=sample)


def test_augmented_dataset_of_large_trusses():
    from python_stable_3d_truss_analysis_b200.generate import GenerateAugmentedDataset

    pool = RO.host_cubes(40, 4, seed=11)
    out = GenerateAugmentedDataset(pool, 64, moveToCentroid=True, noiseStds=(1.0, 1.0, 1.0), seed=3)
    assert (out["info"] == 0).all()
    check_oracle(out, out, 3, names=[0, 1, 2, 3, 63])


def test_order_hook_equals_the_plan_rule():
    cases = fixtures(3) + [(f"cube{nc}_{k}", t._pack()) for nc in (14, 40, 80, 216)
                           for k, t in enumerate(RO.host_cubes(nc, 2, seed=nc))]
    for dim, cs in ((3, cases), (2, fixtures(2))):
        p = pack([t for _, t in cs])
        d = to_dev(p)
        order, env = _lib.ragged_env_order_device(dim, d)
        order, env = order.cpu().numpy(), env.cpu().numpy()
        for b, (name, t) in enumerate(cs):
            want = RO.plan_order(dim, t[1], t[2])
            j0, j1 = int(p["joint_off"][b]), int(p["joint_off"][b + 1])
            assert list(order[j0:j1]) == want["order"], name
            plan = _lib.Plan(dim, np.asarray(t[2], np.int32), np.asarray(t[1], np.uint8))
            assert env[b] == plan.info.envelope_size == want["envelope_size"], name


def _cube7_pool():
    return [tuple(orc.arrays_from_json(json.load(open(f"{H.GOLDEN}/ref_generate/cube-7_case_{i}.json")), 3))
            for i in range(1, 11)]


def test_routing_and_bit_identity():
    small = _cube7_pool()
    big = [t._pack() for t in RO.host_cubes(40, 3, seed=21)]
    # a batch that fits the fused kernels never launches the envelope kernel
    ps = pack(small)
    alone_small, names = run(_lib.solve_ragged_device, 3, ps)
    assert not ran(names, "k_rag_env") and ran(names, "k_dense16")
    # a mixed batch launches both; every truss keeps the bits of its own kernel
    mixed = small[:5] + big[:1] + small[5:] + big[1:]
    which = ["s"] * 5 + ["b"] + ["s"] * 5 + ["b"] * 2
    pm = pack(mixed)
    res, names = run(_lib.solve_ragged_device, 3, pm)
    assert ran(names, "k_rag_env") and ran(names, "k_dense16")
    pb = pack(big)
    alone_big, names_b = run(_lib.solve_ragged_env_device, 3, pb)
    assert ran(names_b, "k_rag_env")
    si = bi = 0
    for b, w in enumerate(which):
        got = rows(res, pm, 3, b)
        want = rows(alone_small, ps, 3, si) if w == "s" else rows(alone_big, pb, 3, bi)
        for k in FIELDS + ("info",):
            assert np.array_equal(got[k], want[k]), (b, w, k)
        si, bi = si + (w == "s"), bi + (w == "b")
    check_oracle(res, pm, 3)


def test_determinism_and_batch_independence():
    torch = _torch()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    pool = [t._pack() for t in RO.host_cubes(20, 6, seed=31)]
    n = 2 * (2 * sms) + 3                                     # two CTAs per SM: every slot used more than twice
    rng = np.random.default_rng(4)
    trusses = []
    for i in range(n):
        xyz, sup, conn, aed, force = pool[i % len(pool)]
        trusses.append((xyz + rng.normal(0, 1.0, xyz.shape), sup, conn, aed, force))
    p = pack(trusses)
    a, _ = run(_lib.solve_ragged_env_device, 3, p)
    b, _ = run(_lib.solve_ragged_env_device, 3, p)
    for k in FIELDS + ("info",):
        assert np.array_equal(a[k], b[k]), k
    assert (a["info"] == 0).all()
    for i in (0, 1, n // 2, n - 1):                           # the same truss alone
        one = pack([trusses[i]])
        r, _ = run(_lib.solve_ragged_env_device, 3, one)
        for k in FIELDS:
            assert np.array_equal(rows(a, p, 3, i)[k], rows(r, one, 3, 0)[k]), (i, k)
    # the same truss at another position of the batch
    rev = pack(trusses[::-1])
    c, _ = run(_lib.solve_ragged_env_device, 3, rev)
    for i in (0, 7, n - 1):
        for k in FIELDS:
            assert np.array_equal(rows(a, p, 3, i)[k], rows(c, rev, 3, n - 1 - i)[k]), (i, k)


def test_failure_classes_among_good_trusses():
    big = [t._pack() for t in RO.host_cubes(40, 2, seed=41)]
    good = big[0]
    xyz, sup, conn, aed, force = good
    bad = {}
    s = sup.copy()
    s[:] = orc.NO                                              # the counting rule (no supports)
    bad[-1] = (xyz, s, conn, aed, force)
    x2 = xyz.copy()
    x2[conn[3, 1]] = x2[conn[3, 0]]                            # a zero-length member
    bad[-2] = (x2, sup, conn, aed, force)
    s3 = sup.copy()
    s3[5] = 9                                                  # an unknown support code
    bad[-3] = (xyz, s3, conn, aed, force)
    c4 = conn.copy()
    c4[7, 0] = len(xyz) + 3                                    # a joint id out of range
    bad[-4] = (xyz, sup, c4, aed, force)
    # singular but passes the counting rule: a joint held by one member only, loaded across it
    free = np.flatnonzero(sup == orc.NO)
    j_new = len(xyz)
    xs = np.vstack([xyz, xyz[free[0]] + np.array([50.0, 0.0, 0.0])])
    ss = np.r_[sup, orc.NO].astype(np.uint8)
    cs = np.vstack([conn, [[free[0], j_new]]]).astype(np.int32)
    as_ = np.vstack([aed, aed[:1]])
    fs = np.r_[force, [0.0, 1000.0, 0.0]]
    bad["singular"] = (xs, ss, cs, as_, fs)
    order = [good, bad[-1], big[1], bad[-2], good, bad[-3], big[1], bad[-4], good, bad["singular"], big[1]]
    kinds = ["g", -1, "g", -2, "g", -3, "g", -4, "g", "singular", "g"]
    p = pack(order)
    ref = pack([t for t, k in zip(order, kinds) if k == "g"])
    for fn in (_lib.solve_ragged_env_device, _lib.solve_ragged_device):
        res, names = run(fn, 3, p)
        assert ran(names, "k_rag_env")
        r0, _ = run(fn, 3, ref)
        gi = 0
        for b, k in enumerate(kinds):
            got = rows(res, p, 3, b)
            if k == "g":
                for f in FIELDS + ("info",):
                    assert np.array_equal(got[f], rows(r0, ref, 3, gi)[f]), (b, f)
                gi += 1
                continue
            info = int(got["info"][0])
            if k == "singular":
                assert info > 0, info
                ordr, _ = _lib.ragged_env_order_device(3, to_dev(pack([bad["singular"]])))
                ordr = ordr.cpu().numpy()
                # k - 1 is the position of the pivot in the elimination order: the new joint's first free DOF
                s_ = bad["singular"][1]
                pos = 0
                for j in ordr:
                    if j == j_new:
                        break
                    pos += int(sum(orc.free_mask(3, s_[j:j + 1])))
                assert info - 1 in (pos, pos + 1, pos + 2), (info, pos)
            else:
                assert info == k, (b, k, info)
            for f in FIELDS:
                assert not np.isnan(got[f]).any() and not np.any(got[f]), (b, f)
    # a truss whose offsets claim more than max_joint: -4 with zero outputs, its neighbours solved as alone
    torch = _torch()
    small_, large_ = sorted(big, key=lambda t: (len(t[0]), len(t[2])))
    assert len(large_[0]) > len(small_[0]) or len(large_[2]) > len(small_[2])
    trio = pack([small_, large_, small_])
    d = to_dev(trio)
    out = _lib.solve_ragged_env_device(3, d, max_joint=len(small_[0]), max_member=len(small_[2]))
    torch.cuda.synchronize()
    out = {k: v.cpu().numpy() for k, v in out.items()}
    alone, _ = run(_lib.solve_ragged_env_device, 3, pack([small_]))
    assert list(out["info"]) == [0, -4, 0]
    assert float(out["weight"][1]) == 0.0
    for b in (0, 2):
        for f in FIELDS:
            assert np.array_equal(rows(out, trio, 3, b)[f], rows(alone, pack([small_]), 3, 0)[f]), (b, f)


def test_host_entry_point_equals_device():
    big = [t._pack() for t in RO.host_cubes(40, 3, seed=51)] + _cube7_pool()[:4]
    p = pack(big)
    host = _lib.solve_ragged_host(3, p["joint_off"], p["member_off"], p["xyz"], p["support"], p["conn"], p["aed"], p["force"])
    dev, _ = run(_lib.solve_ragged_device, 3, p)
    for k in FIELDS + ("info",):
        assert np.array_equal(np.asarray(host[k]), dev[k]), k


def test_scratch_across_streams_and_graphs():
    torch = _torch()
    big = [t._pack() for t in RO.host_cubes(40, 4, seed=61)]
    p = pack(big)
    d = to_dev(p)
    ref = _lib.solve_ragged_device(3, d)
    torch.cuda.synchronize()
    ref = {k: v.cpu().numpy() for k, v in ref.items()}
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    for i in range(4):                                         # alternating streams share the arena
        st = s1 if i % 2 == 0 else s2
        with torch.cuda.stream(st):
            o = _lib.solve_ragged_device(3, d, stream=st)
        st.synchronize()
        for k in FIELDS:
            assert np.array_equal(o[k].cpu().numpy(), ref[k]), (i, k)
    # capture after a warm-up on the capturing stream; replays give the same bits
    gs = torch.cuda.Stream()
    mj, mm = int(np.diff(p["joint_off"]).max()), int(np.diff(p["member_off"]).max())
    out = {k: torch.empty_like(torch.from_numpy(v)).cuda() for k, v in ref.items()}
    with torch.cuda.stream(gs):
        _lib.solve_ragged_device(3, d, out=out, stream=gs, max_joint=mj, max_member=mm)
    gs.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=gs):
        _lib.solve_ragged_device(3, d, out=out, stream=gs, max_joint=mj, max_member=mm)
    for v in out.values():
        v.zero_()
    g.replay()
    torch.cuda.synchronize()
    for k in FIELDS:
        assert np.array_equal(out[k].cpu().numpy(), ref[k]), k
    # a captured call that would grow the arena is refused with nothing enqueued: the same sizes as a warm-up call (the
    # launch configuration is then known), but a batch whose persistent grid needs more slots than any call made so far
    many = pack(big * 160)
    dm = to_dev(many)
    few = pack(big)
    _lib.solve_ragged_device(3, to_dev(few), max_joint=200, max_member=2000)      # warm-up of the sizes, 4 slots
    torch.cuda.synchronize()
    g2 = torch.cuda.CUDAGraph()
    with pytest.raises(_lib.TrussLibError) as ei:
        with torch.cuda.graph(g2, stream=gs):
            _lib.solve_ragged_device(3, dm, stream=gs, max_joint=200, max_member=2000)
    assert ei.value.code == -8                                 # TB_ERR_ALLOC
    torch.cuda.synchronize()
    o = _lib.solve_ragged_device(3, dm, max_joint=200, max_member=2000)   # outside a capture the call grows the arena
    torch.cuda.synchronize()
    o = {k: v.cpu().numpy() for k, v in o.items()}
    for b in (0, 5, len(big) * 160 - 1):
        for k in FIELDS:
            assert np.array_equal(rows(o, many, 3, b)[k], rows(ref, p, 3, b % len(big))[k]), (b, k)
