#!/usr/bin/env python
"""Benchmark of the hot path: FP64 trusses solved / second through the batched Truss.Solve.

    python bench.py --gpus N --steps K --warmup W            # the CUDA path (one rank per GPU under torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host cores (oracle port)

Workload (BASELINE.json configs[1]): the bar-942 truss (tests/golden/ref_data/bar-942_input_0.json) under a batch of
1024 synthetic load cases per GPU (SURVEY.md section 8d recipe: the fixture's loaded joints, components ~ U(-10,10),
default_rng(0)).  Every load case is solved as an independent Truss.Solve(): member geometry, assembly of K_ff, dense
blocked Cholesky, forward/back substitution, recovery of axial forces and reactions -- nothing is shared or skipped
between the systems of a batch (the factor-once / 1024-right-hand-sides shortcut is NOT what is timed here).

One JSON line on stdout (rank 0).  `value` = systems of all ranks / device time (inputs resident in HBM);
`e2e` = same metric through the C ABI's host entry point (tb_solve_host) with pinned host buffers, H2D + D2H inside the
timed region; `roofline` = the dominant kernel (k_band for bar-942) against the FP64 tensor (DMMA) peak measured in this run;
`cpu_baseline` = the oracle port of the reference (numpy, per-member Python loops + LAPACK) on this box's cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FIXTURE = os.path.join(ROOT, "tests", "golden", "ref_data", "bar-942_input_0.json")
BATCH_PER_GPU = 1024
METRIC = "FP64 trusses solved/sec (batched Truss.Solve)"
UNIT = "trusses/s"
WORKLOAD = "bar-942 (n=696 free DOF, 942 members) x 1024 independent load-case solves per GPU, FP64"
# the workload description both arms print (the driver compares the two lines' `config`): nothing arm-specific in here
CONFIG = {"workload": WORKLOAD, "batch_per_gpu": BATCH_PER_GPU, "n_free": 696, "n_member": 942, "mode": "independent K per system",
          "timing": "GPU arm: device time per step (CUDA events), explicit 256 MB L2 flush (> 126 MB L2) between timed steps, "
                    "outside the events; CPU arm: wall clock of a bounded sample of the same load cases on all host cores"}


def load_cases(n_case: int, seed: int = 0):
    """SURVEY.md 8d config 2: keep the fixture's loaded joints, components ~ U(-10,10)."""
    data = json.load(open(FIXTURE))
    loaded = sorted(j for j, v in data["force"] if any(abs(float(x)) >= 1e-10 for x in v))
    rng = np.random.default_rng(seed)
    nj = len(data["joint"])
    F = np.zeros((n_case, nj, 3))
    F[:, loaded, :] = rng.uniform(-10.0, 10.0, size=(n_case, len(loaded), 3))
    return data, F.reshape(n_case, nj * 3)


# ------------------------------------------------------------------------------------------ CPU arm
def _cpu_worker(args):
    os.environ["OPENBLAS_NUM_THREADS"] = "1"
    from oracle import truss_oracle as orc
    dim, arrs, Fs = args
    joints, support, conn, aed = arrs
    out = 0.0
    for f in Fs:
        r = orc.solve(dim, joints, support, conn, aed, f)
        out += float(r["u"][0])
    return out


def cpu_port_throughput(n_solve_per_core: int = 6):
    """Oracle port (reference algorithm: per-member Python loops + LAPACK dgesv) on all host cores."""
    import multiprocessing as mp
    from oracle import truss_oracle as orc

    data, F = load_cases(64)
    joints, support, conn, aed, _ = orc.arrays_from_json(data, 3)
    cores = len(os.sched_getaffinity(0))
    # serial figure first (what one Truss.Solve() loop gives a user today)
    t0 = time.perf_counter()
    orc.solve(3, joints, support, conn, aed, F[0])
    warm = time.perf_counter() - t0
    n_serial = max(3, min(12, int(3.0 / max(warm, 1e-3))))
    t0 = time.perf_counter()
    for i in range(n_serial):
        orc.solve(3, joints, support, conn, aed, F[i % 64])
    serial = n_serial / (time.perf_counter() - t0)
    # all cores: one process per core, OPENBLAS_NUM_THREADS=1
    per = n_solve_per_core
    jobs = [(3, (joints, support, conn, aed), [F[(c * per + i) % 64] for i in range(per)]) for c in range(cores)]
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        pool.map(_cpu_worker, [(3, (joints, support, conn, aed), [F[0]])] * cores)   # warm the workers
        t0 = time.perf_counter()
        pool.map(_cpu_worker, jobs)
        dt = time.perf_counter() - t0
    return {"value": cores * per / dt, "unit": UNIT, "cores": cores, "kind": "port", "sample_solves": cores * per,
            "sample": f"{cores * per} of the 1024 bar-942 load cases, {cores} processes x {per} solves, "
                      f"OPENBLAS_NUM_THREADS=1 (oracle/truss_oracle.py: solve)",
            "serial_value": serial, "serial_sample": f"{n_serial} solves on one core, OpenBLAS default threads"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals = []
    for _ in range(max(1, args.warmup)):
        cpu_port_throughput(2)
    base = None
    for _ in range(max(1, args.steps)):
        base = cpu_port_throughput(6)
        vals.append(base["value"])
    v = float(np.mean(vals))
    base["value"] = v
    # a "step" of this arm is the bounded sample (cores x 6 solves): ms_per_step is its measured wall time; the time the
    # full 1024 x n_gpus batch would take at this rate is reported beside it, never instead of it
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * base["sample_solves"] / v, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": dict(CONFIG),
            "reference_run": {"what": "reference algorithm (oracle port: per-member Python loops + LAPACK dgesv) on the host cores",
                              "solves_per_step": base["sample_solves"],
                              "extrapolated_ms_for_the_full_batch": 1e3 * BATCH_PER_GPU * args.gpus / v},
            "cpu_baseline": base,
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu), "-f", self.path],
                                         stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        try:
            rows = [r.split(",") for r in open(self.path).read().strip().splitlines() if r.strip()]
            sm = [float(r[1]) for r in rows]
            pw = [float(r[3]) for r in rows]
            busy = [s for s, p in zip(sm, pw) if p >= 0.5 * max(pw)] or sm
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            reasons = sorted({n for r in rows for n, v in zip(names, r[5:9]) if v.strip().lower().startswith("active")})
            out = {"sm_mhz": float(np.median(busy)), "sm_max_mhz": float(rows[0][2]), "reasons": reasons,
                   "samples": len(rows), "power_w_max": max(pw)}
        except Exception as exc:  # keep the bench line even if nvidia-smi misbehaves
            out["error"] = str(exc)
        finally:
            try:
                os.unlink(self.path)
            except OSError:
                pass
        return out


# ------------------------------------------------------------------------------------------ GPU arm
def dump_outputs(dirname: str, out: dict):
    """Write what one step returns to its caller, one float64 DIR/<name>.npy per array: u, ext [B, N], axial [B, M],
    weight [B] and the per-system status codes info [B] (0: solved).  For bar-942 x 1024 that is 20 MB."""
    os.makedirs(dirname, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(dirname, name + ".npy"), t.cpu().numpy().astype(np.float64))


def run_gpu(args):
    # libraries (NCCL's version banner) may write to fd 1: keep the real stdout for the one JSON line
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist

    from python_stable_3d_truss_analysis_b200 import _lib
    from python_stable_3d_truss_analysis_b200.truss import Truss

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    B = BATCH_PER_GPU
    data, F_all = load_cases(B * world)
    F = F_all[rank * B:(rank + 1) * B]                      # contiguous block partition (SURVEY.md 8e)
    truss = Truss(3).LoadFromJSON(data=data)
    xyz, support, conn, aed, _ = truss._pack()
    plan = truss._get_plan(support, conn)
    N, M, n = plan.N, plan.M, plan.n

    td = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    d_xyz, d_aed, d_F = td(xyz), td(aed), td(F)
    # one flat result buffer per rank, [u | ext | axial]: the three outputs are views into it.  With several GPUs the
    # results go back to rank 0 (north_star: gather only).  Preferred: rank r's flat buffer IS slice r of a buffer in
    # rank 0's HBM, mapped into every process (symmetric memory over NVLink / NVSwitch), so k_recover's stores are the
    # gather -- compute and transfer in one kernel, one device-side barrier after it.  TB_BENCH_GATHER=nccl (or a
    # failed rendezvous) falls back to a separate NCCL gather of the local flat buffer.
    per_rank = B * (2 * N + M)
    gathered, symm, gather_mode = None, None, "single GPU"
    mode = os.environ.get("TB_BENCH_GATHER", "pipelined")
    pipelined = False
    if world > 1 and mode in ("peer", "pipelined"):
        try:
            from python_stable_3d_truss_analysis_b200.parallel import PeerGather, PipelinedPeerGather
            if mode == "pipelined":
                symm = PipelinedPeerGather(per_rank, torch.float64, dev, dst=0)
                pipelined = True
                flat = symm.bufs[0]
                gather_mode = ("results of step i are pushed into rank 0's buffer (peer-mapped symmetric memory over NVLink) by a copy "
                               "stream while step i+1 computes into a second buffer; one signal barrier after the last step")
            else:
                symm = PeerGather(per_rank, torch.float64, dev, dst=0)
                flat = symm.local                               # my slice of rank 0's buffer
                gather_mode = "k_recover stores straight into rank 0's buffer (peer-mapped symmetric memory over NVLink), one signal barrier"
            gathered = symm.slices
        except Exception as exc:   # noqa: BLE001
            print(f"bench.py: symmetric-memory rendezvous failed ({exc!r}); using the NCCL gather", file=sys.stderr)
            symm, pipelined = None, False
    if symm is None:
        flat = torch.empty(per_rank, dtype=torch.float64, device=dev)
        if world > 1:
            gathered = [torch.empty_like(flat) for _ in range(world)] if rank == 0 else None
            gather_mode = "NCCL gather of u/ext/axial to rank 0 inside the step"
    def views(fl):
        return {"u": fl[:B * N].view(B, N), "ext": fl[B * N:2 * B * N].view(B, N), "axial": fl[2 * B * N:].view(B, M)}

    w_info = {"weight": torch.empty(B, dtype=torch.float64, device=dev), "info": torch.empty(B, dtype=torch.int32, device=dev)}
    out = {**views(flat), **w_info}
    outs2 = [{**views(bf), **w_info} for bf in symm.bufs] if pipelined else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # > 126 MB L2
    stream = torch.cuda.current_stream()
    step_no = [0]

    def step(st=None):
        if pipelined:                          # compute into buffer i & 1; the copy stream ships it while the next step runs
            i = step_no[0]
            step_no[0] += 1
            symm.acquire(i, stream)
            plan.solve_device(B, d_xyz, d_F, aed=d_aed, out=outs2[i & 1], stream=stream)
            symm.submit(i, stream)
            return
        plan.solve_device(B, d_xyz, d_F, aed=d_aed, out=out, stream=stream if st is None else st)
        if symm is not None:
            symm.barrier()                     # every rank's results have landed in rank 0's buffer
        elif world > 1:
            dist.gather(flat, gathered, dst=0)

    def drain():
        if pipelined:
            symm.drain(stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        step()
    drain()
    barrier()
    assert not bool(out["info"].any().item()), "a system failed to factorise"
    if pipelined:
        out = outs2[(step_no[0] - 1) & 1]      # the buffer the last step computed into (parity gate below)

    # ---- multi-GPU: what rank 0 received from the last rank equals what it computes itself for those load cases
    if world > 1 and rank == 0:
        chk = torch.empty(per_rank, dtype=torch.float64, device=dev)
        chk_out = {"u": chk[:B * N].view(B, N), "ext": chk[B * N:2 * B * N].view(B, N), "axial": chk[2 * B * N:].view(B, M),
                   "weight": torch.empty(B, dtype=torch.float64, device=dev), "info": torch.empty(B, dtype=torch.int32, device=dev)}
        plan.solve_device(B, d_xyz, td(F_all[(world - 1) * B:world * B]), aed=d_aed, out=chk_out, stream=stream)
        torch.cuda.synchronize()
        assert torch.equal(chk, gathered[world - 1]), "gathered results of the last rank differ from a local solve"
        del chk, chk_out
    barrier()

    # ---- parity gate on the timed batch (oracle = checker only): 2 sampled systems, 1e-9 norm-wise
    if rank == 0:
        from oracle import truss_oracle as orc
        joints, sup_o, conn_o, aed_o, _ = orc.arrays_from_json(data, 3)
        for b in (0, B - 1):
            want = orc.solve_closed_form(3, joints, sup_o, conn_o, aed_o, F[b])
            for k in ("u", "ext", "axial"):
                err = orc.normwise_err(out[k][b].cpu().numpy(), want[k])
                assert err <= 1e-9, f"parity gate failed: system {b} field {k} err {err:.3e}"

    # ---- timed region: K steps, each timed on the device; L2 flushed between steps (outside the events).  On one GPU the
    # step (three kernel launches through tb_solve) is captured once into a CUDA graph and replayed (TB_BENCH_GRAPH=0:
    # plain launches); the per-kernel times of the roofline come from a second, instrumented pass of K steps.
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = _lib.launch_count()
    step()
    launches_per_step = _lib.launch_count() - launches0
    graph = None
    if world == 1 and os.environ.get("TB_BENCH_GRAPH", "1") == "1":
        try:
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                step(torch.cuda.current_stream())
            graph.replay()
            torch.cuda.synchronize()
        except Exception as exc:   # noqa: BLE001
            print(f"bench.py: CUDA graph capture failed ({exc!r}); plain launches", file=sys.stderr)
            graph = None
            torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    wall0 = time.perf_counter()
    for e0, e1 in ev:
        flush.zero_()
        e0.record(stream)
        if graph is not None:
            graph.replay()
        else:
            step()
        e1.record(stream)
    ev_drain = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    ev_drain[0].record(stream)
    drain()                                    # pipelined gather: the last copies + the signal barrier are part of the timed region
    ev_drain[1].record(stream)
    barrier()
    wall = time.perf_counter() - wall0
    launches = launches_per_step * args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outs2[(step_no[0] - 1) & 1] if pipelined else out)
    # instrumented pass: CUDA events around every kernel (they cost a few microseconds per step, hence not in the timed pass)
    _lib.profile_enable(True)
    _lib.profile_read()
    evp = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for e0, e1 in evp:
        flush.zero_()
        e0.record(stream)
        step()
        e1.record(stream)
    drain()
    barrier()
    prof = _lib.profile_read()
    _lib.profile_enable(False)
    prof_ms = sum(e0.elapsed_time(e1) for e0, e1 in evp)
    # ---- sustained rate: back-to-back steps for --sustain-s seconds (no flush: a step cycles 350 MB of factor / K workspace
    # through the 126 MB L2 on its own), one event pair around the whole run, clocks sampled during it
    sustained = None
    if args.sustain_s > 0:
        n_sus = max(50, int(args.sustain_s / max(1e-6, (sum(e0.elapsed_time(e1) for e0, e1 in ev) / args.steps) * 1e-3)))
        sus_sampler = ClockSampler(local)
        if rank == 0:
            sus_sampler.start()
        barrier()
        es0, es1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        es0.record(stream)
        for _ in range(n_sus):
            if graph is not None:
                graph.replay()
            else:
                step()
        drain()
        es1.record(stream)
        barrier()
        ts_ = torch.tensor([es0.elapsed_time(es1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ts_, op=dist.ReduceOp.MAX)
        sus_clocks = sus_sampler.stop() if rank == 0 else None
        sustained = {"value": B * world * n_sus / (float(ts_.item()) * 1e-3), "unit": UNIT, "seconds": float(ts_.item()) * 1e-3,
                     "steps": n_sus, "ms_per_step": float(ts_.item()) / n_sus, "clocks": sus_clocks,
                     "what": "back-to-back steps without the L2 flush, one CUDA-event pair around the run, max over ranks"}
    dev_ms = sum(e0.elapsed_time(e1) for e0, e1 in ev) + ev_drain[0].elapsed_time(ev_drain[1])
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms = float(t.item())
    ms_per_step = dev_ms / args.steps
    value = B * world / (ms_per_step * 1e-3)

    # ---- same 1024 load cases with the factorisation shared (SURVEY.md 8d asks for both timings): K assembled and
    # factorised once, 1024 substitutions + recoveries (tb_solve_loadcases).  Reported beside the headline, never as it.
    shared = None
    if plan.path == 2 and not args.headline_only:
        flat2 = torch.empty_like(flat)
        out2 = {"u": flat2[:B * N].view(B, N), "ext": flat2[B * N:2 * B * N].view(B, N), "axial": flat2[2 * B * N:].view(B, M),
                "weight": torch.empty(B, dtype=torch.float64, device=dev), "info": torch.empty(B, dtype=torch.int32, device=dev)}
        for _ in range(3):
            plan.solve_device(B, d_xyz, d_F, aed=d_aed, out=out2, stream=stream, shared_factor=True)
        torch.cuda.synchronize()
        worst = max(float((out2[k] - out[k]).abs().max() / out[k].abs().max()) for k in ("u", "ext", "axial"))
        assert worst <= 1e-10, f"shared-factor results differ from the independent ones: {worst:.3e}"
        ev2 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for e0, e1 in ev2:
            flush.zero_()
            e0.record(stream)
            plan.solve_device(B, d_xyz, d_F, aed=d_aed, out=out2, stream=stream, shared_factor=True)
            e1.record(stream)
        torch.cuda.synchronize()
        ms2 = sum(e0.elapsed_time(e1) for e0, e1 in ev2) / args.steps
        shared = {"value": B / (ms2 * 1e-3), "unit": "load cases/s per GPU", "ms_per_step": ms2,
                  "max_rel_diff_vs_independent": worst,
                  "what": "tb_solve_loadcases: one assembly + one factorisation (k_prep, k_band3 on one system), "
                          "k_band_subst (a warp per load case against the shared factor), k_recover"}

    # ---- end to end through the C ABI host entry point: pinned host buffers, H2D + D2H inside the timed region
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()  # noqa: E731
    h_xyz, h_aed, h_F = pin(xyz), pin(aed), pin(F)
    h_out = {"u": pin(np.empty((B, N))), "ext": pin(np.empty((B, N))), "axial": pin(np.empty((B, M))),
             "weight": pin(np.empty(B)), "info": torch.empty(B, dtype=torch.int32).pin_memory().numpy()}
    for _ in range(2):
        plan.solve_host(B, h_xyz, h_F, aed=h_aed, out=h_out)
    barrier()
    e2e_steps = max(3, min(args.steps, 10))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        plan.solve_host(B, h_xyz, h_F, aed=h_aed, out=h_out)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_blocking = B * world * e2e_steps / float(t.item())
    assert np.array_equal(h_out["u"], out["u"].cpu().numpy()), "host and device entry points disagree"
    # the same batches streamed through the pipelined entry point (tb_solve_host_async / tb_host_wait): three batches in
    # flight, so the copies of one batch travel under the kernels of its neighbours; every step still copies its inputs
    # from and its results to pinned host memory inside the timed region, and the region ends when the last result is home.
    # Results come back in the compact layout (u_free [n], react [s], axial [M], weight: everything the dense u / ext /
    # axial hold -- u is zero at supports, ext is the caller's own load vector at free DOFs, truss.py:342-351) and, for
    # comparison, in the dense one.
    free_idx, _, sup_idx = plan.maps()
    want_dev = {"u_free": out["u"][:, torch.from_numpy(free_idx.astype(np.int64)).to(dev)].cpu().numpy(),
                "react": out["ext"][:, torch.from_numpy(sup_idx.astype(np.int64)).to(dev)].cpu().numpy(),
                "u": out["u"].cpu().numpy(), "ext": out["ext"].cpu().numpy(), "axial": out["axial"].cpu().numpy()}
    pin_i32 = lambda n_: torch.empty(n_, dtype=torch.int32).pin_memory().numpy()  # noqa: E731
    pipe_steps = max(e2e_steps, min(4 * args.steps, 60))

    def stream_batches(layout):
        shapes = {"u": (B, N), "ext": (B, N), "axial": (B, M), "weight": (B,), "u_free": (B, plan.n), "react": (B, plan.s)}
        bufs = [dict({k: pin(np.zeros(shapes[k])) for k in layout}, info=pin_i32(B)) for _ in range(3)]
        tk = [plan.solve_host_async(B, h_xyz, h_F, aed=h_aed, want=layout, out=bufs[i % 3])[0] for i in range(3)]
        for t_ in tk:
            plan.host_wait(t_)
        barrier()
        t0 = time.perf_counter()
        inflight = []
        for i in range(pipe_steps):
            inflight.append(plan.solve_host_async(B, h_xyz, h_F, aed=h_aed, want=layout, out=bufs[i % 3])[0])
            if len(inflight) == 3:                  # one batch uploading, one computing, one downloading
                plan.host_wait(inflight.pop(0))
        for t_ in inflight:
            plan.host_wait(t_)
        pipe_s = time.perf_counter() - t0
        tt = torch.tensor([pipe_s], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        for b in bufs:
            for k in layout:
                if k != "weight":
                    assert np.array_equal(b[k], want_dev[k]), f"pipelined host entry point disagrees with the device entry point ({k})"
        return B * world * pipe_steps / float(tt.item()), int(sum(v.nbytes for v in bufs[0].values()))

    e2e_dense, d2h_dense = stream_batches(("u", "ext", "axial", "weight"))
    e2e_value, d2h_compact = stream_batches(("u_free", "react", "axial", "weight"))
    h2d = int(h_xyz.nbytes + h_aed.nbytes + h_F.nbytes)
    d2h = d2h_compact
    clocks = sampler.stop() if rank == 0 else None

    # ---- the other GPU configurations of BASELINE.json (3: GA population, 4: ragged cube-7 batch, 5: cube 12^3), every rank
    configs = {}
    if not args.headline_only:
        import bench_configs
        peak_dmma0, _ = _lib.fp64_peak(1, 8192)
        peak_dfma0, _ = _lib.fp64_peak(0, 8192)
        try:
            hbm0 = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6650.0)
        except Exception:
            hbm0 = 6650.0
        del flush
        torch.cuda.empty_cache()
        flush2 = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        configs = bench_configs.run_configs(torch, dist, rank, world, dev, max(3, min(args.steps, 10)), flush2,
                                            {"dmma": peak_dmma0, "dfma": peak_dfma0, "hbm": hbm0},
                                            which=tuple(args.configs.split(",")))
        del flush2

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (factorisation + triangular solves) against the FP64 tensor peak measured
    # on this GPU.  Algorithmic flops: the dense potrf count of SURVEY.md 8d when the tiled pipeline treats the
    # matrix as dense; the envelope-Cholesky count (fill stays inside the row envelope of K_ff) when the plan
    # exploits the sparsity -- counting the dense n^3/3 for work that is never done would inflate the fraction.
    peak_dmma, _ = _lib.fp64_peak(1, 8192)
    peak_dfma, _ = _lib.fp64_peak(0, 8192)
    path = plan.path
    ts_prog = plan.ts_program() if path == 2 and os.environ.get("TB_BAND_LEGACY") != "1" else None
    kname = {0: "k_dense16", 1: "k_chol", 2: "k_band_ts" if ts_prog else "k_band2"}[path]
    chol_ms, chol_n = prof["small"] if path == 0 else prof["chol"]
    dense_flops = n ** 3 / 3.0 + n ** 2 / 2.0 + n / 6.0 + 2.0 * n * n               # potrf + two triangular solves (SURVEY 8d)
    dense_mode = os.environ.get("TB_DENSE_TILES") == "1" and path == 1
    flops_per_system = dense_flops if dense_mode else float(plan.info.envelope_flops)
    per_launch_s = chol_ms / max(chol_n, 1) * 1e-3
    achieved = B * flops_per_system / per_launch_s / 1e12
    # DRAM traffic of that kernel per launch: an ncu capture (dram__bytes_read.sum + dram__bytes_write.sum) recorded under
    # profiles/ together with the code revision it was taken at; null when there is none for this kernel
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        traffic = tj.get(f"{kname}_dram_bytes_per_launch")
        traffic_src = tj.get(f"{kname}_source")
    kernels = {k: {"ms_per_step": v[0] / args.steps, "launches": v[1]} for k, v in prof.items() if v[1]}
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    hbm_src = "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650"
    nnz = int(plan.info.nnz_lower)
    # HBM view of the same kernel: compulsory bytes = K_ff non-zeros in, load vector in, displacements out
    solve_bytes = B * (nnz * 8 + 2 * n * 8)
    roof_hbm = {"kernel": kname, "bound": "hbm", "achieved": solve_bytes / per_launch_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                "frac": solve_bytes / per_launch_s / 1e9 / hbm_peak, "peak_source": hbm_src,
                "bytes_per_system": nnz * 8 + 2 * n * 8}
    # HBM-bound stages: member products + K_ff values (k_geom + k_kval), recovery (k_recover); SURVEY 8d byte counts
    asm_bytes = B * (M * (2 * 4 + 3 * 8) + plan.nJ * 3 * 8 + plan.nJ + nnz * 8)
    rec_bytes = B * (N * 8 + M * (2 * 4 + 8) + plan.nJ * 3 * 8 + (2 * N + M) * 8)
    stages = {}
    for key, byts in (("assemble", asm_bytes), ("recover", rec_bytes)):
        ms_k, cnt = prof[key]
        if key == "assemble":
            ms_k += prof["geom"][0]
        if cnt:
            gbs = byts / (ms_k / cnt * 1e-3) / 1e9
            stages[key] = {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                           "bytes_per_launch": byts, "ms_per_launch": ms_k / cnt}

    cpu = cpu_port_throughput(6)
    line_extra = {}
    if ts_prog:
        ti = ts_prog["info"]
        executed = 1024.0 * (ti["products"] + ti["solves"])          # two DMMA m8n8k4 (512 flop) per 8x8 block product / solve
        line_extra = {"executed_dmma_flops_per_system": executed, "executed_over_envelope": executed / flops_per_system,
                      "split": {"top_blocks": ti["bT"], "separator_blocks": ti["nS"], "bottom_blocks": ti["nB"],
                                "chain_block_columns": max(ti["bT"], ti["nB"]) + ti["nS"], "block_columns": ti["nblk"]}}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": dict(CONFIG),
        "run": {"pipeline": {0: "fused shared-memory kernel", 1: "tiled 64x64 block-sparse Cholesky",
                             2: "two-sided block-band Cholesky (8x8 DMMA blocks, top-down and bottom-up warps meeting at a separator)" if ts_prog
                             else "block-band Cholesky (16x16 blocks)"}[path],
                "launch": "CUDA graph replay of the step" if graph is not None else "plain stream launches",
                "multi_gpu": "contiguous block partition of the batch; " + gather_mode},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "api": "tb_solve_host_async + tb_host_wait (C ABI), pinned host buffers, three batches in flight (upload / compute / "
                       "download): every step copies its inputs H2D and its results D2H inside the timed region; results in the "
                       "compact layout (u_free [n] | react [s] | axial [M] | weight: the non-redundant content of u / ext / axial)",
                "steps": pipe_steps,
                "dense_layout": {"value": e2e_dense, "unit": UNIT, "d2h_bytes_per_step": d2h_dense,
                                 "api": "same pipeline, results as dense u [N] | ext [N] | axial [M] | weight"},
                "blocking": {"value": e2e_blocking, "unit": UNIT, "steps": e2e_steps, "d2h_bytes_per_step": d2h_dense,
                             "api": "tb_solve_host: one blocking call per step, dense layout (copies of the step not overlapped with other steps)"}},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"kernel": kname + " (block Cholesky + forward/back substitution)", "bound": "tensor",
                     "achieved": achieved, "peak": peak_dmma, "unit": "TFLOP/s", "frac": achieved / peak_dmma,
                     "traffic": traffic, "traffic_source": traffic_src, "flops_per_system": flops_per_system,
                     "flops_model": "dense potrf (SURVEY 8d)" if dense_mode else "envelope Cholesky + two triangular solves (plan.envelope_flops)",
                     "dense_potrf_equivalent_tflops": B * dense_flops / per_launch_s / 1e12,
                     "peak_source": "FP64 DMMA m8n8k4 microbenchmark (tb_fp64_peak) measured in this run; "
                                    "MEASURED_PEAKS.json has no FP64 entry", "peak_dfma": peak_dfma,
                     "share_of_step": chol_ms / prof_ms, **line_extra},
        "roofline_hbm_view": roof_hbm,
        "roofline_stages": stages,
        "kernels": kernels,
        "cpu_baseline": cpu,
        "sustained": sustained,
        "shared_k": shared,
        "configs": configs,
        "wall_s_timed_region": wall,
    }
    sys.stdout.flush()
    os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--sustain-s", type=float, default=2.0, help="seconds of back-to-back steps for the sustained figure (0: skip)")
    ap.add_argument("--configs", default="3,4,5", help="which of the other BASELINE.json configurations to measure as well")
    ap.add_argument("--headline-only", action="store_true",
                    help="skip the shared-factor extra (profiler runs: the launch list then holds the headline step only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step (rank 0's batch) to DIR/<name>.npy; the inputs are "
                         "seeded, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the CUDA path (--impl b200)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
