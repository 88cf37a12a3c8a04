"""Forward vs forward + backward of a ragged batch (tb_solve_ragged + tb_adjoint_ragged) on the GPU:

  cube-7 x 65 536, the config-4 recipe (the live_cube7_aug.json pool tiled with Gaussian joint jitter, sigma 10).

Same method as tools/adjoint_time.py: device time per step from CUDA events, warmed up first, a 256 MB memset between
timed steps (larger than the 126 MB L2), repetitions until the timed window of each measurement is >= 1 s; medians are
reported.  Per-kernel times (k_dense16 / k_small, k_adj_rhs_ragged, k_sens_ragged) come from torch.profiler in a separate
pass.  Prints the card name and power limit with the numbers and writes one JSON line to --out.

    python tools/adjoint_ragged_time.py --out profiles/r04a_adjoint_ragged_time.json
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.adjoint_time import card, time_steps  # noqa: E402

KERNELS = ("k_dense16", "k_small", "k_adj_rhs_ragged", "k_sens_ragged")


def config4_batch(torch, dev, total):
    from python_stable_3d_truss_analysis_b200.truss import Truss
    from tests import helpers as H

    pool = [Truss(3).LoadFromJSON(data={k: g[k] for k in ("joint", "force", "member")}) for g in H.load_json("live_cube7_aug.json")]
    jo, mo, xyz, sup, conn, aed, force, _ = H.ragged_pool_arrays(pool, total)
    td = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    p = {"joint_off": td(jo), "member_off": td(mo), "xyz": td(xyz), "support": td(sup), "conn": td(conn), "aed": td(aed),
         "force": td(force)}
    SJ, SM = int(jo[-1]), int(mo[-1])
    f64 = dict(dtype=torch.float64, device=dev)
    s = {"p": p, "B": total, "maxj": int(np.diff(jo).max()), "maxm": int(np.diff(mo).max()),
         "fwd": {"u": torch.empty(SJ * 3, **f64), "ext": torch.empty(SJ * 3, **f64), "axial": torch.empty(SM, **f64),
                 "weight": torch.empty(total, **f64), "info": torch.empty(total, dtype=torch.int32, device=dev)},
         "res": {"joint_xyz": torch.empty(SJ * 3, **f64), "member_aed": torch.empty(SM * 3, **f64),
                 "force": torch.empty(SJ * 3, **f64), "info": torch.empty(total, dtype=torch.int32, device=dev)},
         "work": torch.empty(SJ * 3, **f64)}
    g = torch.Generator(device=dev).manual_seed(1)
    s["grads"] = {"u": torch.randn(SJ * 3, generator=g, **f64), "ext": torch.randn(SJ * 3, generator=g, **f64),
                  "axial": torch.randn(SM, generator=g, **f64), "weight": torch.randn(total, generator=g, **f64)}
    s["name"] = f"cube-7 x {total} ragged (config-4 recipe)"
    return s


def forward(s):
    from python_stable_3d_truss_analysis_b200 import _lib
    _lib.solve_ragged_device(3, s["p"], out=s["fwd"], max_joint=s["maxj"], max_member=s["maxm"])


def backward(s):
    from python_stable_3d_truss_analysis_b200 import _lib
    _lib.adjoint_ragged_device(3, s["p"], s["fwd"]["u"], s["grads"], s["res"], max_joint=s["maxj"], max_member=s["maxm"],
                               work=s["work"])


def kernel_times(torch, s, steps):
    """Mean device time per launch of the solve and adjoint kernels (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            forward(s)
            backward(s)
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        for k in KERNELS:
            if k in ev.key and not (k == "k_small" and "ragged" in ev.key):
                tot = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
                out[k] = {"ms_per_launch": round(tot / max(ev.count, 1) / 1e3, 4), "launches": int(ev.count)}
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04a_adjoint_ragged_time.json"))
    ap.add_argument("--total", type=int, default=65536)
    ap.add_argument("--window-s", type=float, default=1.0, help="least timed time per measurement")
    ap.add_argument("--min-reps", type=int, default=20)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("adjoint_ragged_time.py measures on a CUDA device; none is available")
    dev = torch.device("cuda:0")
    name, power = card()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)          # > 126 MB L2
    s = config4_batch(torch, dev, args.total)
    for _ in range(3):                                                      # warm-up of both passes
        forward(s)
        backward(s)
    torch.cuda.synchronize()
    info = s["fwd"]["info"].cpu().numpy()
    assert np.array_equal(info, s["res"]["info"].cpu().numpy())
    f_ms, f_n = time_steps(torch, lambda: forward(s), flush, args.window_s, args.min_reps)
    fb_ms, fb_n = time_steps(torch, lambda: (forward(s), backward(s)), flush, args.window_s, args.min_reps)
    b_ms = fb_ms - f_ms
    row = {"shape": s["name"], "solved": int((info == 0).sum()), "forward_ms": round(f_ms, 4),
           "forward_backward_ms": round(fb_ms, 4), "backward_over_forward": round(b_ms / f_ms, 3),
           "ratio": round(fb_ms / f_ms, 3), "reps": [f_n, fb_n]}
    print(f"{s['name']}: forward {f_ms:.3f} ms   forward+backward {fb_ms:.3f} ms   backward/forward {b_ms / f_ms:.2f}")
    forward(s)
    backward(s)
    row["kernel_ms"] = kernel_times(torch, s, 5)
    print(f"per launch: {row['kernel_ms']}")
    rec = {"what": "tb_solve_ragged vs tb_solve_ragged + tb_adjoint_ragged, device time per step (CUDA events, median), "
                   "256 MB L2 flush between steps; backward_over_forward = (forward_backward - forward) / forward; "
                   "kernel_ms: mean per launch from torch.profiler in a separate pass",
           "gpu": name, "power_limit": power, "rows": [row]}
    print(f"card: {name}, power limit {power}")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write(json.dumps(rec) + "\n")
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
