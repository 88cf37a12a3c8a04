"""Shared loaders for the parity fixtures under tests/golden (see make_golden.py)."""
from __future__ import annotations

import glob
import json
import os
import random
import re

import numpy as np

from oracle import truss_oracle as orc

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TOL = 1e-9          # north_star: relative (norm-wise) tolerance on displacements, forces, reactions
FIELDS = ("u", "ext", "axial")


def dim_of(name: str) -> int:
    return 2 if name.startswith(("bar-10_", "bar-47_")) else 3


def shipped_cases():
    """[(name, dim, input_dict, golden dense dict)] for the reference's data/bar-* files."""
    out = []
    for f in sorted(glob.glob(os.path.join(GOLDEN, "ref_data", "*_input_*.json"))):
        name = os.path.basename(f)[:-5]
        dim = dim_of(name)
        data = json.load(open(f))
        gold = json.load(open(f.replace("_input_", "_output_")))
        out.append((name, dim, data, dense_from_output(gold, dim)))
    return out


def dense_from_output(gold: dict, dim: int):
    nj, nm = len(gold["joint"]), len(gold["member"])
    return {"u": orc.dense_from_sparse(gold["displace"], nj, dim),
            "ext": orc.dense_from_sparse(gold["external"], nj, dim),
            "axial": orc.dense_from_sparse(gold["internal"], nm),
            "weight": float(gold["weight"])}


def cube7_shipped():
    out = []
    for f in sorted(glob.glob(os.path.join(GOLDEN, "ref_generate", "cube-7_case_*.json")),
                    key=lambda p: int(p.rsplit("_", 1)[1][:-5])):
        gold = json.load(open(f))
        out.append((os.path.basename(f)[:-5], 3, gold, dense_from_output(gold, 3)))
    return out


def load_json(name):
    return json.load(open(os.path.join(GOLDEN, name)))


def generator_modes():
    """[(label, GenerateRandomCubeTrusses kwargs)] over every generation method x link type x parallel-member rule."""
    from python_stable_3d_truss_analysis_b200.type import GenerateMethod, LinkType

    out = []
    for method in (GenerateMethod.DFS, GenerateMethod.BFS, GenerateMethod.Random):
        for link in (LinkType.LeftBottom_RightTop, LinkType.Cross, LinkType.Random):
            for par in (False, True):
                kw = dict(gridRange=(4, 3, 3), numCubeRange=(2, 5), numEachRange=(1, 2), method=method, linkType=link,
                          isAllowParallel=par, isPrintMessage=False, seed=11, nForceRange=(2, None),
                          memberTypes=[[1., 1e7, 0.1], [2., 2e7, 0.2]])
                out.append((f"method={method} link={link} parallel={par}", kw))
    return out


def ga_stub_evolve(ga_mod, truss_mod, type_mod):
    """GA.Evolve on bar-25 with a deterministic stand-in fitness (no solve), given the ga / truss / type modules of an
    implementation.  The GA operators draw from `random` like ga.py:151-190, so two implementations seeded alike must
    walk the same populations.  Returns [best gene, its fitness info, final population, history] as JSON-ready lists."""
    def stub(self, gene):
        w = float(sum((g + 1) * ((i % 7) + 1) for i, g in enumerate(gene)))
        return w, (gene[0] % 2 == 0), True

    class StubGA(ga_mod.GA):
        GetFitness = stub

    data = json.load(open(os.path.join(GOLDEN, "ref_data", "bar-25_input_0.json")))
    mts = [type_mod.MemberType(i, 1e7, 0.1 * i) for i in range(1, 6)]
    random.seed(3)
    gene, info, pop, history = StubGA(truss_mod.Truss(3).LoadFromJSON(data=data), mts, nIteration=6, nPop=30,
                                      nElite=8).Evolve(False)
    return [list(gene), list(info), [list(p) for p in pop], list(history)]


def assert_close(got: dict, want: dict, tol=TOL, what=""):
    for k in FIELDS:
        err = orc.normwise_err(got[k], want[k])
        assert err <= tol, f"{what} field {k}: norm-wise err {err:.3e} > {tol:g}"
    w = want["weight"]
    assert abs(got["weight"] - w) <= tol * max(1.0, abs(w)), f"{what} weight {got['weight']} vs {w}"


def key_sets_match(dense_got, dense_want, rel=1e-8):
    """SURVEY section 4 trap 2: sparse-dict key sets are only reproducible away from the 1e-10 cutoff."""
    a, b = np.asarray(dense_got).ravel(), np.asarray(dense_want).ravel()
    scale = max(np.abs(b).max(), 1e-300)
    sig = np.abs(b) > rel * scale
    return bool(np.all((np.abs(a[sig]) >= orc.ZERO_EPS) == (np.abs(b[sig]) >= orc.ZERO_EPS)))


def cube_truss(n_side: int, seed: int = 1):
    """Full n^3 cube-truss grid (SURVEY.md 8d config 5: n_side = 12 -> nJ 2197, M 14868, n 6084)."""
    from python_stable_3d_truss_analysis_b200.generate import GenerateRandomCubeTrusses
    from python_stable_3d_truss_analysis_b200.type import LinkType

    ts = GenerateRandomCubeTrusses(gridRange=(n_side,) * 3, numCubeRange=(n_side ** 3,) * 2, numEachRange=(1, 1),
                                   lengthRange=(100, 200), forceRange=[(-1000, 1000)] * 3,
                                   linkType=LinkType.LeftBottom_RightTop, seed=seed, isPrintMessage=False)
    return ts[0]


def ragged_pool_arrays(pool, n_total: int, sigma: float = 10.0, seed: int = 1):
    """Config 4 recipe (SURVEY.md 8d): tile a pool of generated trusses to n_total systems with fresh Gaussian joint
    jitter (AddJointNoise-style, sigma, default_rng(seed)).  Returns the tb_ragged_in arrays + the pool index of each system."""
    packs = [t._pack() for t in pool]
    which = np.arange(n_total) % len(pool)
    nj = np.array([p[0].shape[0] for p in packs])[which]
    nm = np.array([p[2].shape[0] for p in packs])[which]
    joint_off = np.zeros(n_total + 1, np.int64); joint_off[1:] = np.cumsum(nj)
    member_off = np.zeros(n_total + 1, np.int64); member_off[1:] = np.cumsum(nm)
    cat = lambda i, dt: np.concatenate([np.asarray(packs[w][i]).reshape(-1) for w in which]).astype(dt)  # noqa: E731
    xyz = cat(0, np.float64)
    rng = np.random.default_rng(seed)
    xyz = xyz + rng.normal(0.0, sigma, size=xyz.shape)
    return joint_off, member_off, xyz, cat(1, np.uint8), cat(2, np.int32), cat(3, np.float64), cat(4, np.float64), which


def tower(dim, per_level, levels, seed):
    """A lattice tower: `per_level` joints per level on a ring (2D: a ladder), every level braced to the next; the bottom
    level is pinned.  Half-bandwidth of K_ff ~ 2 * dim * per_level, so per_level sweeps the band width."""
    rng = np.random.default_rng(seed)
    joints, members = [], []
    for lv in range(levels):
        for k in range(per_level):
            if dim == 2:
                p = [float(k) * 2.0 + 0.1 * rng.standard_normal(), float(lv) * 1.5]
            else:
                ang = 2 * np.pi * k / per_level
                p = [3.0 * np.cos(ang) + 0.1 * rng.standard_normal(), 3.0 * np.sin(ang) + 0.1 * rng.standard_normal(), 2.0 * lv]
            joints.append([p, "PIN" if lv == 0 else "NO"])
    jid = lambda lv, k: lv * per_level + (k % per_level)
    mt = lambda: [float(rng.uniform(0.5, 2.0)), 1e4, 0.1]
    for lv in range(levels):
        ring = per_level if (dim == 3 and per_level > 2) else per_level - 1
        for k in range(ring):
            if lv > 0:
                members.append([[jid(lv, k), jid(lv, k + 1)], mt()])
        if dim == 3 and per_level > 3 and lv > 0:                  # cross bracing inside the level
            for k in range(per_level - 2):
                members.append([[jid(lv, 0), jid(lv, k + 2)], mt()]) if k + 2 != per_level - 1 or per_level == 4 else None
        if lv + 1 < levels:
            for k in range(per_level):
                members.append([[jid(lv, k), jid(lv + 1, k)], mt()])
                members.append([[jid(lv, k), jid(lv + 1, k + 1)], mt()])
                if dim == 3:
                    members.append([[jid(lv, k + 1), jid(lv + 1, k)], mt()])
    members = [m for m in members if m is not None and m[0][0] != m[0][1]]
    seen, uniq = set(), []
    for m in members:
        key = tuple(sorted(m[0]))
        if key not in seen:
            seen.add(key)
            uniq.append(m)
    forces = [[jid(levels - 1, k), [float(x) for x in rng.uniform(-5, 5, size=dim)]] for k in range(per_level)]
    return {"joint": joints, "force": forces, "member": uniq}


# --------------------------------------------------------------------------- which CUDA kernels ran (GPU tests)
_KERNEL_TAG = re.compile(r"(k_band_ts|k_band[123]|k_prep)(?:<|ILi)(\d+)")


def kernel_tag(name: str):
    """'k_band_ts<7>', 'k_band2<4>' (the band kernels by NB), 'k_prep<3>' (by dim) from a demangled or mangled kernel
    name; None for any other kernel."""
    m = _KERNEL_TAG.search(name)
    return f"{m.group(1)}<{m.group(2)}>" if m else None


def cuda_kernels(fn):
    """Runs fn() under torch.profiler with CUDA activities and synchronises.  Returns (fn's result, {tag: launches})
    for the kernels kernel_tag() names."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    seen = {}
    for ev in prof.events():
        tag = kernel_tag(ev.name)
        if tag is not None:
            seen[tag] = seen.get(tag, 0) + 1
    return res, seen


def band_kernels(seen):
    """The band factorisation kernels among cuda_kernels()' tags."""
    return sorted(t for t in seen if t.startswith("k_band"))


def solve_device_np(plan, B, xyz, aed, force):
    """plan.solve_device on CUDA copies of numpy inputs (leading dimension B, or shared); returns numpy outputs."""
    import torch

    dev = torch.device("cuda:0")
    td = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(dev)  # noqa: E731
    f64 = dict(dtype=torch.float64, device=dev)
    out = {"u": torch.empty(B, plan.N, **f64), "ext": torch.empty(B, plan.N, **f64), "axial": torch.empty(B, plan.M, **f64),
           "weight": torch.empty(B, **f64), "info": torch.empty(B, dtype=torch.int32, device=dev)}
    plan.solve_device(B, td(xyz), td(force), aed=td(aed), out=out)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


def backward_error(dim, joints, support, conn, aed, force, u):
    """Norm-wise backward error of displacements u for K_ff u_f = f_f: |K_ff u_f - f_f|_inf / (|K_ff|_inf |u_f|_inf +
    |f_f|_inf).  A Cholesky solve in binary64 leaves ~1e-16 whatever the conditioning, so this sees errors in a kernel
    that a forward-error tolerance of an ill-conditioned system would let through."""
    K = orc.assemble_K(dim, joints, conn, aed)
    mask = orc.free_mask(dim, support)
    Kff, uf, ff = K[mask][:, mask], np.asarray(u)[mask], np.asarray(force).reshape(-1)[mask]
    return float(np.abs(Kff @ uf - ff).max() / (np.abs(Kff).sum(axis=1).max() * np.abs(uf).max() + np.abs(ff).max()))


_BAND_CHILD = """
import json, sys
import numpy as np
sys.path.insert(0, {root!r})
from tests import band_catalogue as BC
from tests import helpers as H
seen_all = []
for job in json.loads(sys.argv[1]):
    e = BC.get(job["label"])
    plan = BC.plan_for(e)
    plan.set_path(2)
    xyz, aed, F = BC.inputs(plan, e, job["B"], seed=job["seed"])
    lo, hi = job.get("slice", (0, job["B"]))
    out, seen = H.cuda_kernels(lambda: H.solve_device_np(plan, hi - lo, xyz, aed[lo:hi], F[lo:hi]))
    np.savez(job["dst"], **out)
    seen_all.append(seen)
json.dump(seen_all, open(sys.argv[2], "w"))
"""


def run_band_child(tmp_dir, env, jobs):
    """Band-path solves of catalogue entries (tests/band_catalogue.py) in a fresh process with `env` added: the
    switches TB_BAND_LEGACY, TB_BAND_WARPS and TB_LARGE_SPLIT are read once per process.  Each job is {"label", "B",
    "seed"} and optionally "slice": [lo, hi] (solve only systems lo .. hi-1 of the B-system inputs).  Returns
    [(numpy outputs, {kernel tag: launches})] per job."""
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    tag = "_".join(f"{k}{v}" for k, v in sorted(env.items())) or "default"
    jobs = [dict(j, dst=os.path.join(str(tmp_dir), f"{tag}_{i}.npz")) for i, j in enumerate(jobs)]
    seen_path = os.path.join(str(tmp_dir), f"{tag}_kernels.json")
    subprocess.run([sys.executable, "-c", _BAND_CHILD.format(root=root), json.dumps(jobs), seen_path], check=True,
                   env=dict(os.environ, **env), timeout=600)
    seen = json.load(open(seen_path))
    return [(dict(np.load(j["dst"])), s) for j, s in zip(jobs, seen)]
