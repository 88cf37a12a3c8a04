"""Reverse mode of linear buckling (tb_buckling_adjoint) on the GPU, alone and with the static solve's adjoint that
closes the chain through the member forces (tb_adjoint), next to the forward of the same batch (tb_solve, then
tb_buckling under its member forces):

  bar-72 x 8192 sizings (n = 48), 6 factors;
  bar-120 x 4096 sizings (n = 111), 10 factors.

The member properties are explicit rows (a GA population passes type_table[gene]); the cotangent is 1 on every factor.
Device time per call from CUDA events, every shape warmed up first, a 256 MB memset between timed calls (larger than
the 126 MB L2), repetitions until the timed window of each measurement is >= 1 s; medians are reported (the method of
tools/modes_adjoint_time.py).  Per-launch time of k_buckling_sens comes from torch.profiler in a separate pass; the
modes array it reads (B n_modes N doubles) over that time is set against 7.7 TB/s, the HBM3e bandwidth of the B200's
data sheet.  Prints the card name and power limit with the numbers and writes one JSON line to --out.

    python tools/buckling_adjoint_time.py --out profiles/r10a_buckling_adjoint_time.json
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from buckling_time import card, load  # noqa: E402
from modes_time import time_steps  # noqa: E402

HBM_TBPS = 7.7


def shapes(torch, dev):
    td = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev, torch.float64)  # noqa: E731
    rng = np.random.default_rng(0)
    f64 = dict(dtype=torch.float64, device=dev)
    out = []
    plan, xyz, _, _, _, force = load("bar-72_input_0")
    table = np.stack([rng.uniform(0.1, 3.0, 16), np.full(16, 1e7), np.full(16, 0.1)], 1)
    genes = rng.integers(0, 16, size=(8192, plan.M))
    out.append(dict(name="bar-72 x 8192 sizings, 6 factors", plan=plan, B=8192, xyz=td(xyz), aed=td(table[genes]),
                    force=td(force), nm=6))
    plan, xyz, _, _, aed, force = load("bar-120_input_0")
    aedb = np.repeat(aed[None], 4096, axis=0)
    aedb[:, :, 0] *= rng.uniform(0.5, 2.0, size=(4096, plan.M))
    out.append(dict(name="bar-120 x 4096 sizings, 10 factors", plan=plan, B=4096, xyz=td(xyz), aed=td(aedb),
                    force=td(force), nm=10))
    for s in out:
        p, B = s["plan"], s["B"]
        s["st"] = {"u": torch.empty(B, p.N, **f64), "ext": torch.empty(B, p.N, **f64), "axial": torch.empty(B, p.M, **f64),
                   "weight": torch.empty(B, **f64), "info": torch.empty(B, dtype=torch.int32, device=dev)}
        s["bk"] = {"factor": torch.empty(B, s["nm"], **f64), "modes": torch.empty(B, s["nm"], p.N, **f64),
                   "info": torch.empty(B, dtype=torch.int32, device=dev)}
        s["g"] = torch.ones(B, s["nm"], **f64)
        s["bres"] = {"joint_xyz": torch.empty(B, p.nJ, p.dim, **f64), "member_aed": torch.empty(B, p.M, 3, **f64),
                     "axial": torch.empty(B, p.M, **f64)}
        s["sres"] = {"joint_xyz": torch.empty(B, p.nJ, p.dim, **f64), "member_aed": torch.empty(B, p.M, 3, **f64),
                     "force": torch.empty(B, p.N, **f64)}
    return out


def forward(s):
    s["plan"].solve_device(s["B"], s["xyz"], s["force"], aed=s["aed"], out=s["st"])
    s["plan"].buckling_device(s["B"], s["xyz"], s["st"]["axial"], aed=s["aed"], n_modes=s["nm"], out=s["bk"])


def buckling_adjoint(s):
    s["plan"].buckling_adjoint_device(s["B"], s["xyz"], s["aed"], s["st"]["axial"], s["bk"], s["g"], s["bres"])


def backward(s):
    buckling_adjoint(s)
    s["plan"].adjoint_device(s["B"], s["xyz"], s["force"], s["aed"], s["st"]["u"], {"axial": s["bres"]["axial"]},
                             s["sres"])


def kernel_ms(torch, s, steps):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            buckling_adjoint(s)
        torch.cuda.synchronize()
    for ev in prof.key_averages():
        if "k_buckling_sens" in ev.key:
            tot = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
            return round(tot / max(ev.count, 1) / 1e3, 4)
    return None


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10a_buckling_adjoint_time.json"))
    ap.add_argument("--window-s", type=float, default=1.0, help="least timed time per measurement")
    ap.add_argument("--min-reps", type=int, default=20)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("buckling_adjoint_time.py measures on a CUDA device; none is available")

    dev = torch.device("cuda:0")
    name, power = card()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)          # > 126 MB L2
    rows = []
    all_shapes = shapes(torch, dev)
    for s in all_shapes:
        for _ in range(3):
            forward(s)
            backward(s)
        torch.cuda.synchronize()
        assert not s["st"]["info"].any() and not s["bk"]["info"].any(), s["name"]
        assert bool(torch.isfinite(s["sres"]["member_aed"]).all()), s["name"]
        n_crit = int(torch.isfinite(s["bk"]["factor"]).sum())
        a_ms, a_n = time_steps(torch, lambda: buckling_adjoint(s), flush, args.window_s, args.min_reps)
        b_ms, b_n = time_steps(torch, lambda: backward(s), flush, args.window_s, args.min_reps)
        f_ms, f_n = time_steps(torch, lambda: forward(s), flush, args.window_s, args.min_reps)
        p = s["plan"]
        modes_bytes = s["B"] * s["nm"] * p.N * 8
        row = {"shape": s["name"], "n": p.n, "N": p.N, "M": p.M, "B": s["B"], "n_modes": s["nm"],
               "finite_factors": n_crit, "buckling_adjoint_ms": round(a_ms, 4), "full_backward_ms": round(b_ms, 4),
               "forward_ms": round(f_ms, 4), "backward_over_forward": round(b_ms / f_ms, 4),
               "modes_array_mb": round(modes_bytes / 1e6, 2), "reps": [a_n, b_n, f_n]}
        rows.append(row)
        print(f"{s['name']:36s} tb_buckling_adjoint {a_ms:8.3f} ms   + tb_adjoint {b_ms:8.3f} ms   forward {f_ms:8.3f} ms"
              f"   backward / forward {b_ms / f_ms:.4f}")
    for s, row in zip(all_shapes, rows):
        buckling_adjoint(s)
        k = kernel_ms(torch, s, 5)
        row["k_buckling_sens_ms"] = k
        if k:
            row["modes_bytes_per_s_tb"] = round(row["modes_array_mb"] * 1e6 / (k * 1e-3) / 1e12, 3)
            row["share_of_hbm_7_7_tbps"] = round(row["modes_bytes_per_s_tb"] / HBM_TBPS, 4)
        print(f"{s['name']:36s} k_buckling_sens per launch: {k} ms   {row.get('modes_bytes_per_s_tb')} TB/s of the modes "
              f"array ({row.get('share_of_hbm_7_7_tbps')} of 7.7 TB/s)")
    rec = {"what": "tb_buckling_adjoint alone and with tb_adjoint (the full backward through the static solve) vs the "
                   "forward tb_solve + tb_buckling of the same batch, device time per call (CUDA events, median), 256 MB "
                   "L2 flush between calls; cotangent 1 on every factor; k_buckling_sens_ms: mean per launch from "
                   "torch.profiler in a separate pass; modes_bytes_per_s_tb: B n_modes N doubles over that "
                   "kernel time, against the data sheet's 7.7 TB/s",
           "gpu": name, "power_limit": power, "rows": rows}
    print(f"card: {name}, power limit {power}")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write(json.dumps(rec) + "\n")
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
