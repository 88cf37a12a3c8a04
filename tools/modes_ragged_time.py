"""Time the modal analysis of ragged batches (tb_modes_ragged) on the GPU, with the method of tools/modes_time.py: CUDA
events around each call, a 256 MB buffer zeroed between calls (larger than the 126 MB L2), the median over a window of at
least --window-s seconds.  Shapes:
  * cube-7 x 65 536 (the config-4 recipe: a pool of generated trusses tiled with Gaussian joint jitter), 6 modes, lumped
    and consistent, next to tb_solve_ragged of the same batch and scipy.linalg.eigh per truss on the host (a sample,
    scaled to the batch);
  * bar-72 x 8192 perturbed sizings packed ragged next to tb_modes on the plan (the cost of the row-owner assembly);
  * the cube-7 case with max_free left at 0 (bound min(d max_joint, 160)) next to max_free = the largest free-DOF count.
Prints the card name and power limit with the numbers and writes one JSON line to --out.

    python tools/modes_ragged_time.py --out profiles/r08a_modes_ragged_time.json
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.modes_time import card, time_steps  # noqa: E402


def cube7(torch, dev, total):
    from python_stable_3d_truss_analysis_b200.truss import Truss
    from tests import helpers as H

    pool = [Truss(3).LoadFromJSON(data={k: g[k] for k in ("joint", "force", "member")}) for g in H.load_json("live_cube7_aug.json")]
    jo, mo, xyz, sup, conn, aed, force, _ = H.ragged_pool_arrays(pool, total)
    host = {"joint_off": jo, "member_off": mo, "xyz": xyz, "support": sup, "conn": conn, "aed": aed, "force": force}
    return host, {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in host.items()}


def bar72(torch, dev, B):
    from oracle import truss_oracle as orc
    from python_stable_3d_truss_analysis_b200 import _lib
    from tests import helpers as H

    joints, support, conn, aed, _ = orc.arrays_from_json(H.load_json("ref_data/bar-72_input_0.json"), 3)
    rng = np.random.default_rng(0)
    aeds = np.repeat(aed[None], B, axis=0)
    aeds[:, :, 0] *= rng.uniform(0.5, 2.0, size=(B, len(aed)))
    nj, nm = len(joints), len(conn)
    packed = {"joint_off": np.arange(B + 1, dtype=np.int64) * nj, "member_off": np.arange(B + 1, dtype=np.int64) * nm,
              "xyz": np.tile(joints.reshape(-1), B), "support": np.tile(np.asarray(support, np.uint8), B),
              "conn": np.tile(np.asarray(conn, np.int32).reshape(-1), B), "aed": aeds.reshape(-1)}
    td = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    plan = _lib.Plan(3, conn, support)
    return plan, td(joints), td(aeds), {k: td(v) for k, v in packed.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08a_modes_ragged_time.json"))
    ap.add_argument("--window-s", type=float, default=1.0)
    ap.add_argument("--min-reps", type=int, default=5)
    ap.add_argument("--total", type=int, default=65536)
    ap.add_argument("--host-sample", type=int, default=256)
    args = ap.parse_args()

    import torch

    from oracle import modal
    from python_stable_3d_truss_analysis_b200 import _lib

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    dev = torch.device("cuda:0")
    name, power = card()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    rows = []
    T = lambda fn: time_steps(torch, fn, flush, args.window_s, args.min_reps)  # noqa: E731

    host, d = cube7(torch, dev, args.total)
    B = args.total
    mj, mm, nfree = _lib._modes_ragged_sizes(3, d, 6, None, None, None)
    out = _lib.modes_ragged_device(3, d, 6)
    static_out = _lib.solve_ragged_device(3, d)
    s_ms, s_n = T(lambda: _lib.solve_ragged_device(3, d, out=static_out, max_joint=mj, max_member=mm))
    for consistent in (False, True):
        for mf in ((nfree, 0) if not consistent else (nfree,)):
            kw = dict(max_joint=mj, max_member=mm, max_free=mf)
            _lib.modes_ragged_device(3, d, 6, consistent=consistent, out=out, **kw)          # warm-up (grows the scratch)
            ms, n = T(lambda: _lib.modes_ragged_device(3, d, 6, consistent=consistent, out=out, **kw))
            ok = int((out["info"] == 0).sum().item())
            bound = mf if mf else min(3 * mj, 160)
            rows.append({"shape": f"cube-7 x {B}, 6 modes, {'consistent' if consistent else 'lumped'}, max_free={mf} (bound {bound})",
                         "ms": round(ms, 3), "reps": n, "ok": ok, "tb_solve_ragged_ms": round(s_ms, 3),
                         "ratio_to_static": round(ms / s_ms, 2)})
    # scipy per truss on the host, a sample scaled to the batch
    jo, mo = host["joint_off"], host["member_off"]
    t0 = time.perf_counter()
    S = min(args.host_sample, B)
    for b in range(S):
        j0, j1, m0, m1 = int(jo[b]), int(jo[b + 1]), int(mo[b]), int(mo[b + 1])
        modal.modes(3, host["xyz"][3 * j0:3 * j1].reshape(-1, 3), host["support"][j0:j1],
                    host["conn"][2 * m0:2 * m1].reshape(-1, 2), host["aed"][3 * m0:3 * m1].reshape(-1, 3))
    host_s = (time.perf_counter() - t0) / S * B
    rows.append({"shape": f"cube-7 x {B}: oracle.modal.modes (numpy assembly + scipy.linalg.eigh) per truss on the host ({S} sampled, scaled)",
                 "ms": round(host_s * 1e3, 1)})

    plan, xyz, aeds, pk = bar72(torch, dev, 8192)
    res = {"eigval": torch.empty(8192, 6, dtype=torch.float64, device=dev),
           "modes": torch.empty(8192, 6, plan.N, dtype=torch.float64, device=dev),
           "info": torch.empty(8192, dtype=torch.int32, device=dev)}
    rout = _lib.modes_ragged_device(3, pk, 6)
    kw = dict(max_joint=plan.nJ, max_member=plan.M, max_free=plan.n)
    u_ms, u_n = T(lambda: plan.modes_device(8192, xyz, aed=aeds, n_modes=6, out=res))
    r_ms, r_n = T(lambda: _lib.modes_ragged_device(3, pk, 6, out=rout, **kw))
    same = bool(torch.equal(rout["eigval"], res["eigval"]))
    rows.append({"shape": "bar-72 x 8192 sizings, 6 modes, lumped: ragged (tb_modes_ragged) vs uniform (tb_modes)",
                 "ms": round(r_ms, 3), "tb_modes_ms": round(u_ms, 3), "ratio": round(r_ms / u_ms, 3), "same_eigval_bits": same})

    rec = {"tool": "tools/modes_ragged_time.py", "method": "CUDA events per call, median over a >= %.1f s window, 256 MB "
           "flush between calls" % args.window_s, "gpu": name, "power_limit": power, "rows": rows}
    print(f"card: {name}, power limit {power}")
    for r in rows:
        print(r)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as fh:
        fh.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
