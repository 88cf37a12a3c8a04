"""Reverse mode of the modal analysis (tb_modes_adjoint) on the GPU, next to the tb_modes forward of the same batch:

  bar-72 x 8192 sizings (n = 48): 6 modes and all 48, lumped and consistent mass;
  bar-120 x 4096 sizings (n = 111): 10 modes and all 111, lumped mass.

The member properties are explicit rows (a GA population passes type_table[gene]); the cotangent is 1 on every mode, so
no mode is skipped.  Device time per call from CUDA events, every shape warmed up first, a 256 MB memset between timed
calls (larger than the 126 MB L2), repetitions until the timed window of each measurement is >= 1 s; medians are
reported (the method of tools/modes_time.py).  Per-launch time of k_modes_sens comes from torch.profiler in a separate
pass.  The modes array the adjoint reads (B n_modes N doubles) over the kernel time is set against 7.7 TB/s, the HBM3e
bandwidth of the B200's data sheet.  Host arm: the numpy eigval_grad of oracle/modal_adjoint.py per system (eigenpairs
given).  Prints the card name and power limit with the numbers and writes one JSON line to --out.

    python tools/modes_adjoint_time.py --out profiles/r07a_modes_adjoint_time.json
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from modes_time import card, load, time_steps  # noqa: E402

HBM_TBPS = 7.7


def shapes(torch, dev):
    td = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev, torch.float64)  # noqa: E731
    rng = np.random.default_rng(0)
    out = []
    _, plan, xyz, aed, _ = load("bar-72_input_0")
    table = np.stack([rng.uniform(0.1, 3.0, 16), np.full(16, 1e7), np.full(16, 0.1)], 1)
    genes = rng.integers(0, 16, size=(8192, plan.M))
    for nm in (6, plan.n):
        for consistent in (False, True):
            out.append(dict(name=f"bar-72 x 8192, {nm} modes, {'consistent' if consistent else 'lumped'}", plan=plan,
                            B=8192, xyz=td(xyz), aed=td(table[genes]), nm=nm, consistent=consistent))
    _, plan, xyz, aed, _ = load("bar-120_input_0")
    aedb = np.repeat(aed[None], 4096, axis=0)
    aedb[:, :, 0] *= rng.uniform(0.5, 2.0, size=(4096, plan.M))
    for nm in (10, plan.n):
        out.append(dict(name=f"bar-120 x 4096, {nm} modes, lumped", plan=plan, B=4096, xyz=td(xyz), aed=td(aedb), nm=nm,
                        consistent=False))
    for s in out:
        p, B = s["plan"], s["B"]
        f64 = dict(dtype=torch.float64, device=dev)
        s["fwd"] = {"eigval": torch.empty(B, s["nm"], **f64), "modes": torch.empty(B, s["nm"], p.N, **f64),
                    "info": torch.empty(B, dtype=torch.int32, device=dev)}
        s["g"] = torch.ones(B, s["nm"], **f64)
        s["res"] = {"joint_xyz": torch.empty(B, p.nJ, p.dim, **f64), "member_aed": torch.empty(B, p.M, 3, **f64),
                    "joint_mass": torch.empty(B, p.nJ, **f64)}
    return out


def forward(s):
    s["plan"].modes_device(s["B"], s["xyz"], aed=s["aed"], n_modes=s["nm"], consistent=s["consistent"], out=s["fwd"])


def adjoint(s):
    s["plan"].modes_adjoint_device(s["B"], s["xyz"], s["aed"], s["fwd"], s["g"], s["res"], consistent=s["consistent"])


def kernel_ms(torch, s, steps):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            adjoint(s)
        torch.cuda.synchronize()
    for ev in prof.key_averages():
        if "k_modes_sens" in ev.key:
            tot = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
            return round(tot / max(ev.count, 1) / 1e3, 4)
    return None


def host_arm():
    """ms per system of oracle/modal_adjoint.py eigval_grad (numpy, eigenpairs given), all modes and the lowest few."""
    from oracle import modal
    from oracle import modal_adjoint
    from oracle import truss_oracle as orc

    res = {}
    for name, few, count in (("bar-72_input_0", 6, 200), ("bar-120_input_0", 10, 100)):
        data = json.load(open(os.path.join(ROOT, "tests", "golden", "ref_data", name + ".json")))
        joints, support, conn, aed, _ = orc.arrays_from_json(data, 3)
        r = modal.modes(3, joints, support, conn, aed)
        for k in (few, len(r["eigval"])):
            g = np.ones(k)
            t0 = time.perf_counter()
            for _ in range(count):
                modal_adjoint.eigval_grad(3, joints, support, conn, aed, r["eigval"][:k], r["modes"][:k], g)
            res[f"{name[:-8]}, {k} modes"] = round((time.perf_counter() - t0) / count * 1e3, 4)
    res["what"] = "ms per system of oracle/modal_adjoint.py eigval_grad, one process"
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07a_modes_adjoint_time.json"))
    ap.add_argument("--window-s", type=float, default=1.0, help="least timed time per measurement")
    ap.add_argument("--min-reps", type=int, default=20)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("modes_adjoint_time.py measures on a CUDA device; none is available")

    dev = torch.device("cuda:0")
    name, power = card()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)          # > 126 MB L2
    rows = []
    all_shapes = shapes(torch, dev)
    for s in all_shapes:
        for _ in range(3):
            forward(s)
            adjoint(s)
        torch.cuda.synchronize()
        assert not s["fwd"]["info"].any(), s["name"]
        assert bool(torch.isfinite(s["res"]["member_aed"]).all()), s["name"]
        f_ms, f_n = time_steps(torch, lambda: forward(s), flush, args.window_s, args.min_reps)
        a_ms, a_n = time_steps(torch, lambda: adjoint(s), flush, args.window_s, args.min_reps)
        p = s["plan"]
        modes_bytes = s["B"] * s["nm"] * p.N * 8
        row = {"shape": s["name"], "n": p.n, "N": p.N, "M": p.M, "B": s["B"], "n_modes": s["nm"],
               "modes_adjoint_ms": round(a_ms, 4), "modes_forward_ms": round(f_ms, 4), "ratio": round(a_ms / f_ms, 4),
               "modes_array_mb": round(modes_bytes / 1e6, 2), "reps": [a_n, f_n]}
        rows.append(row)
        print(f"{s['name']:36s} adjoint {a_ms:8.3f} ms   forward {f_ms:8.3f} ms   ratio {a_ms / f_ms:.4f}   "
              f"modes array {modes_bytes / 1e6:.1f} MB")
    for s, row in zip(all_shapes, rows):
        adjoint(s)
        k = kernel_ms(torch, s, 5)
        row["k_modes_sens_ms"] = k
        if k:
            row["modes_bytes_per_s_tb"] = round(row["modes_array_mb"] * 1e6 / (k * 1e-3) / 1e12, 3)
            row["share_of_hbm_7_7_tbps"] = round(row["modes_bytes_per_s_tb"] / HBM_TBPS, 4)
        print(f"{s['name']:36s} k_modes_sens per launch: {k} ms   {row.get('modes_bytes_per_s_tb')} TB/s of the modes "
              f"array ({row.get('share_of_hbm_7_7_tbps')} of 7.7 TB/s)")
    t0 = time.time()
    host = host_arm()
    print("host arm:", host, f"({time.time() - t0:.0f} s)")
    rec = {"what": "tb_modes_adjoint vs the tb_modes forward of the same batch, device time per call (CUDA events, "
                   "median), 256 MB L2 flush between calls; cotangent 1 on every mode; k_modes_sens_ms: mean per launch "
                   "from torch.profiler in a separate pass; modes_bytes_per_s_tb: B n_modes N doubles over that kernel "
                   "time, against the data sheet's 7.7 TB/s",
           "gpu": name, "power_limit": power, "rows": rows, "host_eigval_grad": host}
    print(f"card: {name}, power limit {power}")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write(json.dumps(rec) + "\n")
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
