"""Shared loaders for the parity fixtures under tests/golden (see make_golden.py)."""
from __future__ import annotations

import glob
import json
import os
import random

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
