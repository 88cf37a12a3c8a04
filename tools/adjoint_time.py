"""Forward vs forward + backward (tb_solve + tb_adjoint) on the GPU for three shapes:

  bar-942 x 1024 independent systems (the bench's headline shape, one factorisation per load case),
  bar-942 x 1024 load cases with shared_factor (one factorisation, 1024 substitutions, in both passes),
  bar-72 x 8192 random sizings (the GA-sized fused path).

Device time per step from CUDA events, every shape warmed up first, a 256 MB memset between timed steps (larger than
the 126 MB L2, as bench.py), repetitions until the timed window of each measurement is >= 1 s; medians are reported.
Per-kernel times of k_adj_rhs / k_sens come from torch.profiler in a separate pass.  Prints the card name and power
limit with the numbers and writes one JSON line to --out.

    python tools/adjoint_time.py --out profiles/r03a_adjoint_time.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
    except Exception:
        import torch
        name, power = torch.cuda.get_device_name(0), "unknown"
    return name, power


def shapes(torch, dev):
    from python_stable_3d_truss_analysis_b200.truss import Truss

    gold = os.path.join(ROOT, "tests", "golden", "ref_data")
    out = []
    rng = np.random.default_rng(0)
    td = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(dev)  # noqa: E731
    t = Truss(3).LoadFromJSON(os.path.join(gold, "bar-942_input_0.json"))
    xyz, _, _, aed, _ = t._pack()
    plan = t._get_plan()
    F = rng.uniform(-10.0, 10.0, size=(1024, plan.N))
    for shared in (False, True):
        out.append(dict(name="bar-942 x 1024" + (" shared_factor" if shared else " independent"), plan=plan, B=1024,
                        xyz=td(xyz), aed=td(aed), force=td(F), shared=shared))
    t = Truss(3).LoadFromJSON(os.path.join(gold, "bar-72_input_0.json"))
    xyz, _, _, aed, force = t._pack()
    plan = t._get_plan()
    aedb = np.repeat(aed[None], 8192, axis=0)
    aedb[:, :, 0] = rng.uniform(0.1, 5.0, size=(8192, plan.M))
    out.append(dict(name="bar-72 x 8192 sizings", plan=plan, B=8192, xyz=td(xyz), aed=td(aedb), force=td(force), shared=False))
    for s in out:
        p, B = s["plan"], s["B"]
        f64 = dict(dtype=torch.float64, device=dev)
        s["fwd"] = {"u": torch.empty(B, p.N, **f64), "ext": torch.empty(B, p.N, **f64), "axial": torch.empty(B, p.M, **f64),
                    "weight": torch.empty(B, **f64), "info": torch.empty(B, dtype=torch.int32, device=dev)}
        g = torch.Generator(device=dev).manual_seed(1)
        s["grads"] = {"u": torch.randn(B, p.N, generator=g, **f64), "ext": torch.randn(B, p.N, generator=g, **f64),
                      "axial": torch.randn(B, p.M, generator=g, **f64), "weight": torch.randn(B, generator=g, **f64)}
        s["res"] = {"joint_xyz": torch.empty(B, p.nJ, p.dim, **f64), "member_aed": torch.empty(B, p.M, 3, **f64),
                    "force": torch.empty(B, p.N, **f64), "info": torch.empty(B, dtype=torch.int32, device=dev)}
    return out


def forward(s):
    s["plan"].solve_device(s["B"], s["xyz"], s["force"], aed=s["aed"], out=s["fwd"], shared_factor=s["shared"])


def backward(s):
    s["plan"].adjoint_device(s["B"], s["xyz"], s["force"], s["aed"], s["fwd"]["u"], s["grads"], s["res"],
                             shared_factor=s["shared"])


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


def kernel_times(torch, s, steps):
    """Mean device time per launch of the two adjoint kernels (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            forward(s)
            backward(s)
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        for k in ("k_adj_rhs", "k_sens"):
            if k in ev.key:
                tot = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
                out[k] = round(tot / max(ev.count, 1) / 1e3, 4)          # us -> ms
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03a_adjoint_time.json"))
    ap.add_argument("--window-s", type=float, default=1.0, help="least timed time per measurement")
    ap.add_argument("--min-reps", type=int, default=20)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("adjoint_time.py measures on a CUDA device; none is available")
    dev = torch.device("cuda:0")
    name, power = card()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)          # > 126 MB L2
    rows = []
    for s in shapes(torch, dev):
        for _ in range(3):                                                  # warm-up of every shape and both passes
            forward(s)
            backward(s)
        torch.cuda.synchronize()
        assert not s["res"]["info"].any(), s["name"]
        f_ms, f_n = time_steps(torch, lambda: forward(s), flush, args.window_s, args.min_reps)
        fb_ms, fb_n = time_steps(torch, lambda: (forward(s), backward(s)), flush, args.window_s, args.min_reps)
        rows.append({"shape": s["name"], "forward_ms": round(f_ms, 4), "forward_backward_ms": round(fb_ms, 4),
                     "ratio": round(fb_ms / f_ms, 3), "reps": [f_n, fb_n]})
        print(f"{s['name']:32s} forward {f_ms:8.3f} ms   forward+backward {fb_ms:8.3f} ms   ratio {fb_ms / f_ms:5.2f}")
    # per-kernel times in a separate, profiled pass
    for s, row in zip(shapes(torch, dev), rows):
        forward(s)
        backward(s)
        row["kernel_ms"] = kernel_times(torch, s, 5)
        print(f"{s['name']:32s} per launch: {row['kernel_ms']}")
    rec = {"what": "tb_solve vs tb_solve + tb_adjoint, device time per step (CUDA events, median), 256 MB L2 flush "
                   "between steps; kernel_ms: mean per launch from torch.profiler in a separate pass",
           "gpu": name, "power_limit": power, "rows": rows}
    print(f"card: {name}, power limit {power}")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write(json.dumps(rec) + "\n")
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
