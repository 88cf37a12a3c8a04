"""Ragged batches beyond the fused kernels on the GPU (tb_solve_ragged -> k_rag_env):

  generated cube-20 x 16384, cube-40 x 8192, cube-80 x 2048, cube-216 x 512 (grid 6^3, tb_gencube on the device);
  the config-4 recipe (cube-7 x 65 536, live_cube7_aug.json tiled with Gaussian jitter) with 1 % cube-40 mixed in,
  against the pure cube-7 batch.

Same method as tools/adjoint_time.py: device time per step from CUDA events, warmed up first, a 256 MB memset between
timed steps (larger than the 126 MB L2), repetitions until the timed window of each measurement is >= 1 s; medians are
reported.  Per-kernel times come from torch.profiler in a separate pass.  Envelope flops: the order hook
(tb_ragged_env_order) gives every truss's envelope; its flops (the count tb_plan_create reports as envelope_flops) are
computed from the restated order of a sample of trusses whose envelope sizes must equal the hook's, and scaled to the
batch by the mean.  The DFMA peak (tb_fp64_peak), the card name and the power limit are read in the same run.  For the
cube-40 row, today's per-topology fallback (one plan and one tb_solve per truss) is timed on 64 trusses, wall time
including the host plan.

    python tools/ragged_env_time.py --out profiles/r05a_ragged_env_time.json
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

from tools.adjoint_time import card, time_steps  # noqa: E402

KERNELS = ("k_rag_env", "k_dense16", "k_small")
SAMPLE = 48


def generated(torch, num_cube, n, seed):
    from python_stable_3d_truss_analysis_b200 import _lib
    from python_stable_3d_truss_analysis_b200.generate import GenerateRandomCubeTrussesOnDevice

    g = GenerateRandomCubeTrussesOnDevice(n, gridRange=(6, 6, 6), numCubeRange=(num_cube, num_cube), lengthRange=(100, 200),
                                          isDoStructuralAnalysis=False, seed=seed, asNumpy=False)
    assert int((g["gen_info"] != 0).sum()) == 0
    return {k: g[k] for k in ("joint_off", "member_off", "xyz", "support", "conn", "aed", "force")}, _lib


def config4(torch, dev, total, mix_cube40):
    from python_stable_3d_truss_analysis_b200.truss import Truss
    from tests import helpers as H

    pool = [Truss(3).LoadFromJSON(data={k: g[k] for k in ("joint", "force", "member")}) for g in H.load_json("live_cube7_aug.json")]
    jo, mo, xyz, sup, conn, aed, force, _ = H.ragged_pool_arrays(pool, total)
    p = {"joint_off": jo, "member_off": mo, "xyz": xyz, "support": sup, "conn": conn, "aed": aed, "force": force}
    if mix_cube40:
        from tests import ragged_order as RO
        big = [t._pack() for t in RO.host_cubes(40, 8, seed=7)]
        n40 = total // 100
        trusses = []
        for b in range(total):
            j0, j1, m0, m1 = jo[b], jo[b + 1], mo[b], mo[b + 1]
            trusses.append((xyz[3 * j0:3 * j1], sup[j0:j1], conn[2 * m0:2 * m1], aed[3 * m0:3 * m1], force[3 * j0:3 * j1]))
        step = total // n40
        for i in range(n40):                                   # spread over the batch
            trusses[i * step] = tuple(np.asarray(a).reshape(-1) for a in big[i % len(big)])
        nj = np.array([len(t[1]) for t in trusses])
        nm = np.array([len(t[2]) // 2 for t in trusses])
        jo, mo = np.zeros(total + 1, np.int64), np.zeros(total + 1, np.int64)
        jo[1:], mo[1:] = np.cumsum(nj), np.cumsum(nm)
        cat = lambda i, dt: np.concatenate([np.asarray(t[i], dt).reshape(-1) for t in trusses])  # noqa: E731
        p = {"joint_off": jo, "member_off": mo, "xyz": cat(0, np.float64), "support": cat(1, np.uint8),
             "conn": cat(2, np.int32), "aed": cat(3, np.float64), "force": cat(4, np.float64)}
    return {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in p.items()}


def outputs(torch, p):
    SJ, SM, B = int(p["support"].numel()), int(p["conn"].numel()) // 2, int(p["joint_off"].numel()) - 1
    f64 = dict(dtype=torch.float64, device=p["xyz"].device)
    return {"u": torch.empty(SJ * 3, **f64), "ext": torch.empty(SJ * 3, **f64), "axial": torch.empty(SM, **f64),
            "weight": torch.empty(B, **f64), "info": torch.empty(B, dtype=torch.int32, device=p["xyz"].device)}


def envelope_flops(lib, p):
    """(sum of envelope entries over the batch from the order hook, estimated envelope flops of the batch)."""
    from tests import ragged_order as RO

    order, env = lib.ragged_env_order_device(3, p)
    env = env.cpu().numpy()
    jo, mo = p["joint_off"].cpu().numpy(), p["member_off"].cpu().numpy()
    sup, conn = p["support"].cpu().numpy(), p["conn"].cpu().numpy()
    B = len(jo) - 1
    idx = np.linspace(0, B - 1, min(SAMPLE, B)).astype(int)
    fl = []
    for b in idx:
        r = RO.plan_order(3, sup[jo[b]:jo[b + 1]], conn[2 * mo[b]:2 * mo[b + 1]])
        assert r["envelope_size"] == env[b], (b, r["envelope_size"], env[b])
        fl.append(r["envelope_flops"])
    return int(env.sum()), float(np.mean(fl)) * B


def kernel_times(torch, fn, steps):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        for k in KERNELS:
            if k in ev.key and not (k == "k_small" and "ragged" in ev.key):
                tot = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
                out[k] = {"ms_per_launch": round(tot / max(ev.count, 1) / 1e3, 4), "launches": int(ev.count)}
    return out


def fallback_per_truss(torch, lib, p, n=64):
    """Today's route for distinct large topologies: one plan (host) and one tb_solve per truss; wall ms per truss."""
    jo, mo = p["joint_off"].cpu().numpy(), p["member_off"].cpu().numpy()
    h = {k: p[k].cpu().numpy() for k in ("xyz", "support", "conn", "aed", "force")}
    dev = p["xyz"].device
    items = []
    for b in range(n):
        j0, j1, m0, m1 = jo[b], jo[b + 1], mo[b], mo[b + 1]
        items.append((h["conn"][2 * m0:2 * m1].reshape(-1, 2), h["support"][j0:j1],
                      torch.from_numpy(h["xyz"][3 * j0:3 * j1].copy()).to(dev), torch.from_numpy(h["aed"][3 * m0:3 * m1].copy()).to(dev),
                      torch.from_numpy(h["force"][3 * j0:3 * j1].copy()).to(dev)))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for conn, sup, xyz, aed, force in items:
        plan = lib.Plan(3, conn, sup)
        f64 = dict(dtype=torch.float64, device=dev)
        out = {"u": torch.empty(1, plan.N, **f64), "info": torch.empty(1, dtype=torch.int32, device=dev)}
        plan.solve_device(1, xyz, force, aed=aed, out=out)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / n


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05a_ragged_env_time.json"))
    ap.add_argument("--scale", type=float, default=1.0, help="batch sizes times this (rehearsals)")
    ap.add_argument("--window-s", type=float, default=1.0, help="least timed time per measurement")
    ap.add_argument("--min-reps", type=int, default=10)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("ragged_env_time.py measures on a CUDA device; none is available")
    from python_stable_3d_truss_analysis_b200 import _lib

    dev = torch.device("cuda:0")
    name, power = card()
    peak_tflops, _ = _lib.fp64_peak(0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)          # > 126 MB L2
    rows = []
    cases = [(f"generated cube-{nc} x {int(n * args.scale)}", "gen", nc, int(n * args.scale))
             for nc, n in ((20, 16384), (40, 8192), (80, 2048), (216, 512))]
    cases += [(f"config-4 cube-7 x {int(65536 * args.scale)}", "c4", 0, int(65536 * args.scale)),
              (f"config-4 cube-7 x {int(65536 * args.scale)} + 1 % cube-40", "c4mix", 0, int(65536 * args.scale))]
    for label, kind, nc, n in cases:
        if kind == "gen":
            p, _ = generated(torch, nc, n, seed=nc)
        else:
            p = config4(torch, dev, n, kind == "c4mix")
        B = int(p["joint_off"].numel()) - 1
        mj = int((p["joint_off"][1:] - p["joint_off"][:-1]).max())
        mm = int((p["member_off"][1:] - p["member_off"][:-1]).max())
        out = outputs(torch, p)
        step = lambda: _lib.solve_ragged_device(3, p, out=out, max_joint=mj, max_member=mm)  # noqa: E731
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        info = out["info"].cpu().numpy()
        ms, reps = time_steps(torch, step, flush, args.window_s, args.min_reps)
        env_entries, flops = envelope_flops(_lib, p)
        row = {"shape": label, "trusses": B, "max_joint": mj, "max_member": mm, "solved": int((info == 0).sum()),
               "ms": round(ms, 4), "reps": reps, "trusses_per_s": round(B / ms * 1e3, 1),
               "envelope_entries": env_entries, "envelope_flops_est": flops,
               "envelope_gflops_per_s": round(flops / ms / 1e6, 2),
               "share_of_dfma_peak": round(flops / ms / 1e9 / peak_tflops, 5)}
        row["kernel_ms"] = kernel_times(torch, step, 3)
        if kind == "gen" and nc == 40:
            row["fallback_plan_plus_solve_ms_per_truss"] = round(fallback_per_truss(torch, _lib, p), 3)
        print(json.dumps(row))
        rows.append(row)
        del p, out
        torch.cuda.empty_cache()
    rec = {"what": "tb_solve_ragged on batches beyond the fused kernels; device time per step (CUDA events, median over "
                   ">= 1 s), 256 MB L2 flush between steps; envelope flops = the count of tb_plan_create's envelope_flops, "
                   f"mean of {SAMPLE} sampled trusses (their envelope sizes checked against the order hook) times the batch; "
                   "share_of_dfma_peak = envelope flops/s over tb_fp64_peak(DFMA) of the same run; kernel_ms: mean per launch "
                   "from torch.profiler in a separate pass; fallback: Plan + tb_solve per truss, wall time incl. the host plan",
           "gpu": name, "power_limit": power, "dfma_peak_tflops": round(peak_tflops, 3), "rows": rows}
    print(f"card: {name}, power limit {power}, DFMA peak {peak_tflops:.2f} TFLOP/s")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
