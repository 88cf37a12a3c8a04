"""Linear buckling (tb_buckling) on the GPU, next to consistent-mass tb_modes on the same batch (the same eigen-solve,
steps 2-5) and the static call that produces the member forces:

  bar-72 x 8192 GA genes (n = 48), 6 factors, next to tb_fitness (with the axial output) of the genes;
  bar-120 x 4096 sizings (n = 111), 10 factors, next to tb_solve of the sizings.

Device time per call from CUDA events, every shape warmed up first, a 256 MB memset between timed calls (larger than the
126 MB L2), repetitions until the timed window of each measurement is >= 1 s; medians are reported, the two eigen
calls and the static call measured alternately.  Host arm: oracle.buckling per design (both matrices assembled in
Python, scipy.linalg.eigh(K_G_ff, K_ff)) on a sample of designs, scaled to the batch.  Prints the card name and power
limit with the numbers and writes one JSON line to --out.

    python tools/buckling_time.py --out profiles/r09a_buckling_time.json
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
    xyz, support, conn, aed, force = t._pack()
    return t._get_plan(), xyz, support, conn, aed, force


def shapes(torch, dev):
    td = lambda a, dt=torch.float64: torch.from_numpy(np.ascontiguousarray(a)).to(dev, dt)  # noqa: E731
    rng = np.random.default_rng(0)
    f64 = dict(dtype=torch.float64, device=dev)
    out = []
    plan, xyz, sup, conn, aed, force = load("bar-72_input_0")
    table = np.stack([rng.uniform(0.1, 3.0, 16), np.full(16, 1e7), np.full(16, 0.1)], 1)
    genes = rng.integers(0, 16, size=(8192, plan.M)).astype(np.int32)
    out.append(dict(name="bar-72 x 8192 genes, 6 factors", plan=plan, B=8192, xyz=td(xyz), gene=td(genes, torch.int32),
                    table=td(table), aed=None, force=td(force), nm=6, static="tb_fitness",
                    host=(xyz, sup, conn, table[genes[:32]], force)))
    plan, xyz, sup, conn, aed, force = load("bar-120_input_0")
    aedb = np.repeat(aed[None], 4096, axis=0)
    aedb[:, :, 0] *= rng.uniform(0.5, 2.0, size=(4096, plan.M))
    out.append(dict(name="bar-120 x 4096 sizings, 10 factors", plan=plan, B=4096, xyz=td(xyz), gene=None, table=None,
                    aed=td(aedb), force=td(force), nm=10, static="tb_solve", host=(xyz, sup, conn, aedb[:16], force)))
    for s in out:
        p, B = s["plan"], s["B"]
        s["fwd"] = {"u": torch.empty(B, p.N, **f64), "ext": torch.empty(B, p.N, **f64), "axial": torch.empty(B, p.M, **f64),
                    "weight": torch.empty(B, **f64), "info": torch.empty(B, dtype=torch.int32, device=dev),
                    "fitness": torch.empty(B, **f64), "flags": torch.empty(B, 2, dtype=torch.uint8, device=dev)}
        s["bk"] = {"factor": torch.empty(B, s["nm"], **f64), "modes": torch.empty(B, s["nm"], p.N, **f64),
                   "info": torch.empty(B, dtype=torch.int32, device=dev)}
        s["md"] = {"eigval": torch.empty(B, s["nm"], **f64), "modes": torch.empty(B, s["nm"], p.N, **f64),
                   "info": torch.empty(B, dtype=torch.int32, device=dev)}
    return out


def static(s):
    f = s["fwd"]
    if s["static"] == "tb_fitness":
        s["plan"].fitness_device(s["B"], s["xyz"], s["force"], s["gene"], s["table"], 1e30, 1e30,
                                 {"fitness": f["fitness"], "flags": f["flags"], "info": f["info"], "axial": f["axial"]})
    else:
        s["plan"].solve_device(s["B"], s["xyz"], s["force"], aed=s["aed"],
                               out={k: f[k] for k in ("u", "ext", "axial", "weight", "info")})


def buckling(s):
    s["plan"].buckling_device(s["B"], s["xyz"], s["fwd"]["axial"], aed=s["aed"], gene=s["gene"], type_table=s["table"],
                              n_modes=s["nm"], out=s["bk"])


def modes(s):
    s["plan"].modes_device(s["B"], s["xyz"], aed=s["aed"], gene=s["gene"], type_table=s["table"], n_modes=s["nm"],
                           consistent=True, out=s["md"])


def time_alternating(torch, fns, flush, window_s, min_reps):
    """Median ms per call of every function, called in turn (one call each per round) until each has a >= window_s window."""
    ms = [[] for _ in fns]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    while min(len(m) for m in ms) < min_reps or min(sum(m) for m in ms) < window_s * 1e3:
        for i, fn in enumerate(fns):
            flush.zero_()
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            ms[i].append(e0.elapsed_time(e1))
    return [float(np.median(m)) for m in ms], [len(m) for m in ms]


def host_arm(s):
    """ms per design of oracle.buckling (assembly in Python + scipy eigh), sampled."""
    from oracle import buckling as bk
    from oracle import truss_oracle as orc

    xyz, sup, conn, aeds, force = s["host"]
    xyz, conn = xyz.reshape(-1, 3), conn.reshape(-1, 2)
    axs = [orc.solve(3, xyz, sup, conn, a, force)["axial"] for a in aeds]
    bk.buckling(3, xyz, sup, conn, aeds[0], axs[0], n_modes=s["nm"])
    t0 = time.perf_counter()
    for a, ax in zip(aeds, axs):
        bk.buckling(3, xyz, sup, conn, a, ax, n_modes=s["nm"])
    return (time.perf_counter() - t0) / len(aeds) * 1e3


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09a_buckling_time.json"))
    ap.add_argument("--window-s", type=float, default=1.0, help="least timed time per measurement")
    ap.add_argument("--min-reps", type=int, default=20)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("buckling_time.py measures on a CUDA device; none is available")

    dev = torch.device("cuda:0")
    name, power = card()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)          # > 126 MB L2
    rows = []
    for s in shapes(torch, dev):
        for _ in range(3):
            static(s)
            buckling(s)
            modes(s)
        torch.cuda.synchronize()
        assert not s["fwd"]["info"].any() and not s["bk"]["info"].any() and not s["md"]["info"].any(), s["name"]
        n_crit = int(torch.isfinite(s["bk"]["factor"][:, 0]).sum())
        (b_ms, m_ms, s_ms), reps = time_alternating(torch, [lambda: buckling(s), lambda: modes(s), lambda: static(s)],
                                                    flush, args.window_s, args.min_reps)
        h_ms = host_arm(s)
        row = {"shape": s["name"], "n": s["plan"].n, "B": s["B"], "tb_buckling_ms": round(b_ms, 4),
               "tb_modes_consistent_ms": round(m_ms, 4), s["static"] + "_ms": round(s_ms, 4),
               "buckling_over_modes": round(b_ms / m_ms, 3), "buckling_over_static": round(b_ms / s_ms, 2),
               "systems_with_a_critical_factor": n_crit, "host_oracle_ms_per_design": round(h_ms, 4),
               "host_oracle_ms_batch_scaled": round(h_ms * s["B"], 1), "reps": reps}
        rows.append(row)
        print(f"{s['name']:36s} tb_buckling {b_ms:8.3f} ms   tb_modes (consistent) {m_ms:8.3f} ms   x{b_ms / m_ms:5.2f}   "
              f"{s['static']} {s_ms:7.3f} ms   host {h_ms:.2f} ms/design ({h_ms * s['B'] / 1e3:.1f} s per batch)")
    rec = {"what": "tb_buckling vs consistent-mass tb_modes (same steps 2-5) and the static call of the same batch, "
                   "device time per call (CUDA events, median, calls alternated), 256 MB L2 flush between calls; host arm: "
                   "oracle/buckling.py per design (numpy assembly + scipy.linalg.eigh), sampled and scaled to the batch",
           "gpu": name, "power_limit": power, "rows": rows}
    print(f"card: {name}, power limit {power}")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write(json.dumps(rec) + "\n")
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
