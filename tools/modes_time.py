"""Batched modal analysis (tb_modes) on the GPU, next to the static solve of the same batch:

  bar-72 x 8192 GA genes (n = 48): 6 modes and all 48, lumped and consistent mass, next to tb_fitness of the genes;
  bar-120 x 4096 sizings (n = 111): 10 modes and all 111, lumped mass, next to tb_solve of the sizings.

Device time per call from CUDA events, every shape warmed up first, a 256 MB memset between timed calls (larger than the
126 MB L2), repetitions until the timed window of each measurement is >= 1 s; medians are reported.  Per-launch time of
k_modes comes from torch.profiler in a separate pass.  Work per system is counted as (4/3 + 4/3 + 3) n^3 flops
(Householder tridiagonalisation, accumulation of Q, implicit QL with vectors) and set against the DFMA peak that
tb_fp64_peak measures in the same run.  Host arm: scipy.linalg.eigh(K_ff, M_ff) on one core and on all cores (matrices
built beforehand, only eigh timed).  Also records the largest relative eigenvalue error against the oracle per fixture.
Prints the card name and power limit with the numbers and writes one JSON line to --out.

    python tools/modes_time.py --out profiles/r06a_modes_time.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, "tests", "golden", "ref_data")


def flops_per_system(n: int) -> float:
    """tred2 (4/3 n^3) + accumulation of Q (4/3 n^3) + tql2 with vectors (~3 n^3)."""
    return (4.0 / 3.0 + 4.0 / 3.0 + 3.0) * n ** 3


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
    except Exception:
        import torch
        name, power = torch.cuda.get_device_name(0), "unknown"
    return name, power


def load(name):
    from python_stable_3d_truss_analysis_b200.truss import Truss

    t = Truss(3).LoadFromJSON(os.path.join(GOLD, name + ".json"))
    xyz, _, _, aed, force = t._pack()
    return t, t._get_plan(), xyz, aed, force


def shapes(torch, dev):
    td = lambda a, dt=torch.float64: torch.from_numpy(np.ascontiguousarray(a)).to(dev, dt)  # noqa: E731
    rng = np.random.default_rng(0)
    out = []
    _, plan, xyz, aed, force = load("bar-72_input_0")
    table = np.stack([rng.uniform(0.1, 3.0, 16), np.full(16, 1e7), np.full(16, 0.1)], 1)
    genes = rng.integers(0, 16, size=(8192, plan.M)).astype(np.int32)
    for nm in (6, plan.n):
        for consistent in (False, True):
            out.append(dict(name=f"bar-72 x 8192 genes, {nm} modes, {'consistent' if consistent else 'lumped'}", plan=plan,
                            B=8192, xyz=td(xyz), gene=td(genes, torch.int32), table=td(table), aed=None, force=td(force),
                            nm=nm, consistent=consistent, static="tb_fitness"))
    _, plan, xyz, aed, force = load("bar-120_input_0")
    aedb = np.repeat(aed[None], 4096, axis=0)
    aedb[:, :, 0] *= rng.uniform(0.5, 2.0, size=(4096, plan.M))
    for nm in (10, plan.n):
        out.append(dict(name=f"bar-120 x 4096 sizings, {nm} modes, lumped", plan=plan, B=4096, xyz=td(xyz), gene=None,
                        table=None, aed=td(aedb), force=td(force), nm=nm, consistent=False, static="tb_solve"))
    for s in out:
        p, B = s["plan"], s["B"]
        f64 = dict(dtype=torch.float64, device=dev)
        s["res"] = {"eigval": torch.empty(B, s["nm"], **f64), "modes": torch.empty(B, s["nm"], p.N, **f64),
                    "info": torch.empty(B, dtype=torch.int32, device=dev)}
        s["fwd"] = {"u": torch.empty(B, p.N, **f64), "ext": torch.empty(B, p.N, **f64), "axial": torch.empty(B, p.M, **f64),
                    "weight": torch.empty(B, **f64), "info": torch.empty(B, dtype=torch.int32, device=dev),
                    "fitness": torch.empty(B, **f64), "flags": torch.empty(B, 2, dtype=torch.uint8, device=dev)}
    return out


def modes(s):
    s["plan"].modes_device(s["B"], s["xyz"], aed=s["aed"], gene=s["gene"], type_table=s["table"], n_modes=s["nm"],
                           consistent=s["consistent"], out=s["res"])


def static(s):
    if s["static"] == "tb_fitness":
        s["plan"].fitness_device(s["B"], s["xyz"], s["force"], s["gene"], s["table"], 1e30, 1e30,
                                 {"fitness": s["fwd"]["fitness"], "flags": s["fwd"]["flags"], "info": s["fwd"]["info"]})
    else:
        s["plan"].solve_device(s["B"], s["xyz"], s["force"], aed=s["aed"], out={k: s["fwd"][k] for k in
                                                                                ("u", "ext", "axial", "weight", "info")})


def time_steps(torch, fn, flush, window_s, min_reps):
    ms = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    while len(ms) < min_reps or sum(ms) < window_s * 1e3:
        flush.zero_()
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return float(np.median(ms)), len(ms)


def kernel_ms(torch, s, steps):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            modes(s)
        torch.cuda.synchronize()
    for ev in prof.key_averages():
        if "k_modes" in ev.key:
            tot = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
            return round(tot / max(ev.count, 1) / 1e3, 4)
    return None


def accuracy():
    """Largest |lambda - lambda_ref| / lambda_ref over all modes, per fixture and mass model (with and without joint
    masses), tb_modes_host against oracle/modal.py."""
    from oracle import modal
    from oracle import truss_oracle as orc
    from python_stable_3d_truss_analysis_b200 import _lib
    from tests import helpers as H

    cases = [(n, d, data) for n, d, data, _ in H.shipped_cases() if not n.startswith("bar-942")] + \
        [(n, d, data) for n, d, data, _ in H.cube7_shipped()[:2]]
    rows = {}
    for name, dim, data in cases:
        joints, support, conn, aed, _ = orc.arrays_from_json(data, dim)
        plan = _lib.Plan(dim, conn, support)
        jm = np.linspace(0.0, 3.0, len(joints)) * float(np.mean(modal.member_masses(dim, joints, conn, aed)))
        worst = {}
        for consistent in (False, True):
            err = 0.0
            for j in (None, jm):
                ref = modal.modes(dim, joints, support, conn, aed, consistent=consistent, joint_mass=j)["eigval_all"]
                got = plan.modes_host(1, joints, aed=aed, consistent=consistent, joint_mass=j, want_modes=False)["eigval"][0]
                err = max(err, float(np.max(np.abs(got - ref) / np.abs(ref))))
            worst["consistent" if consistent else "lumped"] = err
        rows[name] = {"n": plan.n, **worst}
    return rows


HOST_ARM = r"""
import json, sys, time, numpy as np, scipy.linalg as sl
sys.path.insert(0, sys.argv[1])
from oracle import modal, truss_oracle as orc
out = {}
for name, count in (("bar-72_input_0", 64), ("bar-120_input_0", 16)):
    data = json.load(open(f"{sys.argv[1]}/tests/golden/ref_data/{name}.json"))
    joints, support, conn, aed, _ = orc.arrays_from_json(data, 3)
    K, M, _ = modal.reduced(3, joints, support, conn, aed)
    rng = np.random.default_rng(0)
    mats = [(K * s, M) for s in rng.uniform(0.5, 2.0, count)]
    sl.eigh(*mats[0])
    t0 = time.perf_counter()
    for k, m in mats:
        sl.eigh(k, m)
    out[name] = (time.perf_counter() - t0) / count * 1e3
print(json.dumps(out))
"""


def host_arm():
    res = {}
    for label, env in (("one_core", {"OMP_NUM_THREADS": "1", "OPENBLAS_NUM_THREADS": "1", "MKL_NUM_THREADS": "1"}),
                       ("all_cores", {})):
        e = dict(os.environ)
        for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
            e.pop(k, None)
        e.update(env)
        r = subprocess.run([sys.executable, "-c", HOST_ARM, ROOT], capture_output=True, text=True, env=e, timeout=1800)
        res[label] = {k: round(v, 4) for k, v in json.loads(r.stdout.strip().splitlines()[-1]).items()} if r.returncode == 0 \
            else {"error": r.stderr[-400:]}
    res["cores"] = os.cpu_count()
    res["what"] = "ms per system of scipy.linalg.eigh(K_ff, M_ff), all eigenpairs, lumped mass"
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06a_modes_time.json"))
    ap.add_argument("--window-s", type=float, default=1.0, help="least timed time per measurement")
    ap.add_argument("--min-reps", type=int, default=20)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("modes_time.py measures on a CUDA device; none is available")
    from python_stable_3d_truss_analysis_b200 import _lib

    dev = torch.device("cuda:0")
    name, power = card()
    dfma_tflops = _lib.fp64_peak(0)[0]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)          # > 126 MB L2
    rows = []
    for s in shapes(torch, dev):
        for _ in range(3):
            modes(s)
            static(s)
        torch.cuda.synchronize()
        assert not s["res"]["info"].any(), s["name"]
        m_ms, m_n = time_steps(torch, lambda: modes(s), flush, args.window_s, args.min_reps)
        s_ms, s_n = time_steps(torch, lambda: static(s), flush, args.window_s, args.min_reps)
        n = s["plan"].n
        fl = flops_per_system(n) * s["B"]
        row = {"shape": s["name"], "n": n, "B": s["B"], "modes_ms": round(m_ms, 4), s["static"] + "_ms": round(s_ms, 4),
               "ratio": round(m_ms / s_ms, 2), "systems_per_s": round(s["B"] / m_ms * 1e3, 1),
               "mflop_per_system": round(flops_per_system(n) / 1e6, 4),
               "share_of_dfma_peak": round(fl / (m_ms * 1e-3) / (dfma_tflops * 1e12), 4), "reps": [m_n, s_n]}
        rows.append(row)
        print(f"{s['name']:44s} modes {m_ms:8.3f} ms   {s['static']} {s_ms:7.3f} ms   x{m_ms / s_ms:6.1f}   "
              f"{row['systems_per_s']:.3g} systems/s   {100 * row['share_of_dfma_peak']:.2f} % of DFMA peak")
    for s, row in zip(shapes(torch, dev), rows):
        modes(s)
        row["k_modes_ms"] = kernel_ms(torch, s, 5)
        print(f"{s['name']:44s} k_modes per launch: {row['k_modes_ms']} ms")
    acc = accuracy()
    for k, v in acc.items():
        print(f"{k:28s} n={v['n']:4d}  max rel eigenvalue error: lumped {v['lumped']:.2e}  consistent {v['consistent']:.2e}")
    t0 = time.time()
    host = host_arm()
    print("host arm:", host, f"({time.time() - t0:.0f} s)")
    rec = {"what": "tb_modes vs the static solve of the same batch, device time per call (CUDA events, median), 256 MB L2 "
                   "flush between calls; k_modes_ms: mean per launch from torch.profiler in a separate pass; flops "
                   "(4/3 + 4/3 + 3) n^3 per system against the DFMA peak measured by tb_fp64_peak in this run",
           "gpu": name, "power_limit": power, "dfma_peak_tflops": round(dfma_tflops, 3), "rows": rows,
           "accuracy_max_rel_eigenvalue_error": acc, "host_eigh": host}
    print(f"card: {name}, power limit {power}, DFMA peak {dfma_tflops:.2f} TFLOP/s")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write(json.dumps(rec) + "\n")
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
