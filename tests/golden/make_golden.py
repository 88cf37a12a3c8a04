"""Regenerate the committed parity fixtures.  Runs ONLY in the build container
(needs the read-only reference at /root/reference); the GPU box uses the
committed outputs.

    python tests/golden/make_golden.py

Writes, next to this file:
  ref_data/bar-*_{input,output}_*.json   verbatim copies of the reference's shipped known-answer DATA files
                                         (data/, produced by example.py:124-172 upstream)
  ref_generate/cube-7_case_*.json        verbatim copies of generate/cube-7_case_{1..10}.json (example.py:208-231)
  live_solve.json        the live reference's Truss.Solve() on every ref_data input (dense vectors), this container's numpy
  live_ga_bar72.json     GA.GetFitness (ga.py:139-149) on bar-72 for seeded genes / member types (SURVEY 8d config 3 recipe)
  live_loadcases_bar942.npz  bar-942 under seeded load cases (SURVEY 8d config 2 recipe), live Solve() results
  live_random.json       seeded random 2D/3D trusses (all support types, parallel members, loads on supports), live results
  live_cube7_aug.json    generator + full augmentation list (example.py:239-267 recipe, 7 cubes), live results
  live_cube7_seed42.json GenerateRandomCubeTrusses(seed=42) inputs as regenerated today (must equal ref_generate inputs)
  live_kmatrix.npz       GetKMatrix (non-zeros as <case>.i / .j / .v) and the unknown-displacement DOFs (<case>.free) of
                         every ref_data input
  live_generate_modes.json.gz  GenerateRandomCubeTrusses in every method / link type / parallel rule (helpers.generator_modes)
  live_ga_stub_bar25.json   GA.Evolve on bar-25 with a stand-in fitness (helpers.ga_stub_evolve)

The last three were first written by running live_reference_checks() over this package's own truss / generate / ga /
type modules in place of the reference's, at a revision (d711202) whose tests compared exactly these results with the
live reference and passed; live_reference_checks(ref_shim.load()) rewrites them from the reference itself.
"""
from __future__ import annotations

import glob
import gzip
import json
import os
import random
import shutil
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import ref_shim  # noqa: E402

REF = ref_shim.REFERENCE_ROOT
DIM_OF = {"bar-10": 2, "bar-47": 2}


def dim_of(name: str) -> int:
    return DIM_OF.get(name.split("_")[0], 3)


def tolist(d):
    return {k: (v.tolist() if isinstance(v, np.ndarray) else v) for k, v in d.items()}


def copy_shipped():
    os.makedirs(os.path.join(HERE, "ref_data"), exist_ok=True)
    os.makedirs(os.path.join(HERE, "ref_generate"), exist_ok=True)
    for f in sorted(glob.glob(os.path.join(REF, "data", "*.json"))):
        shutil.copyfile(f, os.path.join(HERE, "ref_data", os.path.basename(f)))
    for f in sorted(glob.glob(os.path.join(REF, "generate", "cube-7_case_*.json"))):
        shutil.copyfile(f, os.path.join(HERE, "ref_generate", os.path.basename(f)))


def live_solve(ref):
    out = {}
    for f in sorted(glob.glob(os.path.join(REF, "data", "*_input_*.json"))):
        name = os.path.basename(f)[:-5]
        t = ref.truss.Truss(dim_of(name)).LoadFromJSON(f)
        t.Solve()
        out[name] = tolist(ref_shim.dense_results(t))
    json.dump(out, open(os.path.join(HERE, "live_solve.json"), "w"))


def live_ga(ref, n_gene=96):
    # SURVEY.md 8d config 3: random.seed(0); typeList per example.py:186; genes per ga.py:151-153
    random.seed(0)
    types = [ref.type.MemberType(i, random.uniform(1e7, 3e7), random.uniform(0.1, 1.0)) for i in range(1, 21)]
    out = {"type_table": [t.Serialize() for t in types], "allow_stress": 30000.0, "allow_displace": 10.0, "cases": {}}
    for case in ("bar-72_input_0", "bar-72_input_1", "bar-120_input_0", "bar-25_input_0"):
        truss = ref.truss.Truss(3).LoadFromJSON(os.path.join(REF, "data", case + ".json"))
        ga = ref.ga.GA(truss, types, 30000.0, 10.0)
        genes = [random.choices(range(20), k=truss.nMember) for _ in range(n_gene)]
        # a few extreme genes so both violation branches are exercised
        genes += [[0] * truss.nMember, [19] * truss.nMember, [i % 20 for i in range(truss.nMember)]]
        fits = [ga.GetFitness(g) for g in genes]
        out["cases"][case] = {"genes": genes, "fitness": [float(f[0]) for f in fits],
                              "stress_ok": [bool(f[1]) for f in fits], "displace_ok": [bool(f[2]) for f in fits]}
    # tighter limits: force the penalty branches
    truss = ref.truss.Truss(3).LoadFromJSON(os.path.join(REF, "data", "bar-72_input_0.json"))
    ga = ref.ga.GA(truss, types, 500.0, 0.02)
    genes = [random.choices(range(20), k=truss.nMember) for _ in range(32)]
    fits = [ga.GetFitness(g) for g in genes]
    out["tight"] = {"case": "bar-72_input_0", "allow_stress": 500.0, "allow_displace": 0.02, "genes": genes,
                    "fitness": [float(f[0]) for f in fits], "stress_ok": [bool(f[1]) for f in fits],
                    "displace_ok": [bool(f[2]) for f in fits]}
    json.dump(out, open(os.path.join(HERE, "live_ga_bar72.json"), "w"))


def loadcases_bar942(n_case):
    """SURVEY.md 8d config 2: keep the fixture's loaded joints, components ~ U(-10,10), default_rng(0)."""
    data = json.load(open(os.path.join(REF, "data", "bar-942_input_0.json")))
    loaded = sorted(j for j, v in data["force"] if any(abs(float(x)) >= 1e-10 for x in v))
    rng = np.random.default_rng(0)
    nj = len(data["joint"])
    F = np.zeros((n_case, nj, 3))
    F[:, loaded, :] = rng.uniform(-10.0, 10.0, size=(n_case, len(loaded), 3))
    return data, F.reshape(n_case, nj * 3)


def live_loadcases(ref, n_case=6):
    data, F = loadcases_bar942(n_case)
    U, E, A = [], [], []
    for b in range(n_case):
        d = dict(data)
        d["force"] = [[j, F[b, 3 * j:3 * j + 3].tolist()] for j in range(len(data["joint"]))]
        t = ref.truss.Truss(3).LoadFromJSON(data=d)
        t.Solve()
        r = ref_shim.dense_results(t)
        U.append(r["u"]); E.append(r["ext"]); A.append(r["axial"])
    np.savez_compressed(os.path.join(HERE, "live_loadcases_bar942.npz"), F=F, u=np.array(U), ext=np.array(E), axial=np.array(A))


def random_truss(rng: random.Random, dim: int, nj: int):
    """A seeded, well-posed random truss: a triangulated strip/tower plus extra (possibly parallel)
    members, every support type, loads on free AND supported joints."""
    pts = []
    for j in range(nj):
        base = [3.0 * (j // 2), 2.0 * (j % 2), 1.5 * ((j // 3) % 2)][:dim]
        pts.append([b + rng.uniform(-0.4, 0.4) for b in base])
    sup_pool = ["PIN", "ROLLER_X", "ROLLER_Y"] + (["ROLLER_Z"] if dim == 3 else [])
    sup = ["NO"] * nj
    sup[0] = "PIN"
    sup[1] = "PIN"
    sup[2] = "PIN" if dim == 3 else rng.choice(sup_pool)
    for j in range(3, nj):
        if rng.random() < 0.15:
            sup[j] = rng.choice(sup_pool)
    members = []
    for j in range(nj):
        for k in range(j + 1, min(nj, j + (5 if dim == 3 else 4))):
            members.append([j, k])
    for _ in range(max(2, nj // 3)):                       # parallel duplicates + reversed orientation
        a, b = rng.choice(members)
        members.append([b, a] if rng.random() < 0.5 else [a, b])
    mts = [[rng.choice([0.5, 1.0, 2.5, 7.0]), rng.choice([1e4, 2.1e5, 1e7, 3e7]), rng.uniform(0.1, 8.0)] for _ in members]
    forces = []
    for j in range(nj):
        r = rng.random()
        if r < 0.45:
            forces.append([j, [rng.uniform(-1e3, 1e3) for _ in range(dim)]])
        elif r < 0.5:
            forces.append([j, [0.0] * dim])                  # dropped by AddExternalForce (truss.py:181)
    return {"joint": [[p, s] for p, s in zip(pts, sup)], "force": forces, "member": [[m, t] for m, t in zip(members, mts)]}


def live_random(ref):
    rng = random.Random(1234)
    cases = []
    for dim in (2, 3):
        for nj in (4, 5, 7, 9, 12, 17, 24, 33, 40):
            for _ in range(2):
                data = random_truss(rng, dim, nj)
                t = ref.truss.Truss(dim).LoadFromJSON(data=data)
                try:
                    t.Solve()
                except Exception as exc:  # singular / unstable draws are skipped, deterministically
                    print("skip", dim, nj, type(exc).__name__)
                    continue
                r = ref_shim.dense_results(t)
                if not np.all(np.isfinite(r["u"])) or np.abs(r["u"]).max() > 1e6:
                    print("skip ill-conditioned", dim, nj)
                    continue
                cases.append({"dim": dim, "data": data, "result": tolist(r)})
    json.dump(cases, open(os.path.join(HERE, "live_random.json"), "w"))
    print("live_random:", len(cases), "cases")


def live_cube7(ref, n_aug=48):
    g = ref.generate
    # (a) the shipped recipe, example.py:208-231 -- inputs must reproduce bit-identically
    lst = g.GenerateRandomCubeTrusses(gridRange=(5, 5, 5), numCubeRange=(7, 7), numEachRange=(1, 10), lengthRange=(100, 200),
                                      forceRange=[(-1000, 1000)] * 3, isDoStructuralAnalysis=True, isPlotTruss=False,
                                      isPrintMessage=False, saveFolder=None, seed=42)
    json.dump([t.Serialize() for t in lst], open(os.path.join(HERE, "live_cube7_seed42.json"), "w"))
    # (b) SURVEY.md 8d config 4 recipe: full augmentation list (example.py:239-267), 7 cubes
    aug = g.TrussDataAugmenterList(g.NoChange(), g.MoveToCentroid(), g.RandomTranslation(translateRange=[-30., 30.]),
                                   g.AddJointNoise(noiseMeans=[0., 0., 0.], noiseStds=[10., 10., 10.]),
                                   g.RandomResetPin(minNumPin=5, maxNumPinRatio=0.6))
    lst = g.GenerateRandomCubeTrusses(gridRange=(5, 5, 5), numCubeRange=(7, 7), numEachRange=(1, n_aug), lengthRange=(100, 200),
                                      forceRange=[(-1000, 1000)] * 3, isDoStructuralAnalysis=True, isPlotTruss=False,
                                      isPrintMessage=False, saveFolder=None, seed=42, augmenter=aug)
    json.dump([t.Serialize() for t in lst], open(os.path.join(HERE, "live_cube7_aug.json"), "w"))


def live_reference_checks(ref):
    from tests import helpers as H

    kmat = {}
    for f in sorted(glob.glob(os.path.join(HERE, "ref_data", "*_input_*.json"))):
        name = os.path.basename(f)[:-5]
        t = ref.truss.Truss(dim_of(name)).LoadFromJSON(f)
        K = t.GetKMatrix()
        i, j = np.nonzero(K)
        kmat.update({name + ".i": i.astype(np.int32), name + ".j": j.astype(np.int32), name + ".v": K[i, j],
                     name + ".free": np.nonzero(t.GetDisplacementUnknownMask())[0].astype(np.int32)})
    np.savez_compressed(os.path.join(HERE, "live_kmatrix.npz"), **kmat)
    modes = {label: [t.Serialize() for t in ref.generate.GenerateRandomCubeTrusses(**kw)] for label, kw in H.generator_modes()}
    with gzip.open(os.path.join(HERE, "live_generate_modes.json.gz"), "wt") as f:
        json.dump(modes, f)
    json.dump(H.ga_stub_evolve(ref.ga, ref.truss, ref.type), open(os.path.join(HERE, "live_ga_stub_bar25.json"), "w"))


def main():
    ref = ref_shim.load()
    copy_shipped()
    live_solve(ref)
    live_ga(ref)
    live_loadcases(ref)
    live_random(ref)
    live_cube7(ref)
    live_reference_checks(ref)
    print("done")


if __name__ == "__main__":
    main()
