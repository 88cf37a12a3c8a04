"""The *_host entry points share their staging arenas: the plan's arena for the uniform calls and a per-device arena for
the ragged ones.  A call that needs more than the arena holds regrows it.  Here several host entry points run in turn on
one plan, each on a larger batch than the one before, so every call regrows the arena that the previous call used.
Each result must equal the matching device entry point's on the same inputs, bit for bit."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import truss_oracle as orc
from python_stable_3d_truss_analysis_b200 import _lib
from tests import helpers as H

pytestmark = pytest.mark.gpu

K = 6                      # modes / buckling factors per system
# Batch sizes grow 4x from call to call, and the per-system staging bytes of these calls differ by less than 1.5x (bar-72:
# 3.9 KB for the gene-table modes call up to 5.7 KB for buckling; 4.8 / 5.9 KB per ragged solve / modes truss), so each
# call needs more than the previous growth left (an eighth more than that call needed).
GROWTH = 4


def bar72():
    return orc.arrays_from_json(json.load(open(f"{H.GOLDEN}/ref_data/bar-72_input_0.json")), 3)


def batch(B, seed):
    """Per-system inputs of B jittered bar-72 designs: joints [B, nJ*3], member properties [B, M*3], loads [B, N]."""
    joints, _, _, aed, force = bar72()
    rng = np.random.default_rng(seed)
    xyz = joints.reshape(1, -1) + rng.normal(0.0, 1.0, size=(B, joints.size))
    props = aed.reshape(1, -1) * (1.0 + 0.2 * rng.random((B, aed.size)))
    loads = force.reshape(1, -1) * (1.0 + rng.random((B, 1)))
    return np.ascontiguousarray(xyz), np.ascontiguousarray(props), np.ascontiguousarray(loads)


def cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def numpy_of(out):
    import torch
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items() if v is not None}


def assert_same(host, dev, keys):
    for k in keys:
        assert host[k].dtype == dev[k].dtype and np.array_equal(host[k].reshape(dev[k].shape), dev[k]), k


def test_uniform_host_calls_share_a_growing_staging_arena():
    _, support, conn, _, _ = bar72()
    plan = _lib.Plan(3, conn, support)
    B = 64

    xyz, aed, _ = batch(B, 1)                                           # modal analysis, consistent mass
    host = plan.modes_host(B, xyz, aed=aed, n_modes=K, consistent=True)
    dev = numpy_of(plan.modes_device(B, cuda(xyz), aed=cuda(aed), n_modes=K, consistent=True,
                                     out={"modes": cuda(np.empty((B, K, plan.N)))}))
    assert np.all(host["info"] == 0)
    assert_same(host, dev, ("eigval", "modes", "info"))

    B *= GROWTH                                                          # static solve
    xyz, aed, force = batch(B, 2)
    host = plan.solve_host(B, xyz, force, aed=aed)
    dev = H.solve_device_np(plan, B, xyz, aed, force)
    assert np.all(host["info"] == 0)
    assert_same(host, dev, ("u", "ext", "axial", "weight", "info"))

    B *= GROWTH                                                          # buckling under the member forces of a solve
    xyz, aed, force = batch(B, 3)
    axial = H.solve_device_np(plan, B, xyz, aed, force)["axial"]
    host = plan.buckling_host(B, xyz, axial, aed=aed, n_modes=K)
    dev = numpy_of(plan.buckling_device(B, cuda(xyz), cuda(axial), aed=cuda(aed), n_modes=K,
                                        out={"modes": cuda(np.empty((B, K, plan.N)))}))
    assert np.all(host["info"] == 0) and np.isfinite(host["factor"]).any()
    assert_same(host, dev, ("factor", "modes", "info"))

    B *= GROWTH                                                          # modal analysis again: genes, lumped mass
    rng = np.random.default_rng(4)
    xyz, _, _ = batch(B, 4)
    table = np.array([[a, 1e7, 0.1] for a in (0.5, 1.0, 2.0, 4.0)])
    gene = rng.integers(0, len(table), size=(B, plan.M), dtype=np.int32)
    jm = rng.random((B, plan.nJ))
    host = plan.modes_host(B, xyz, gene=gene, type_table=table, n_modes=K, joint_mass=jm)
    dev = numpy_of(plan.modes_device(B, cuda(xyz), gene=cuda(gene), type_table=cuda(table), n_modes=K, joint_mass=cuda(jm),
                                     out={"modes": cuda(np.empty((B, K, plan.N)))}))
    assert np.all(host["info"] == 0)
    assert_same(host, dev, ("eigval", "modes", "info"))


def ragged_growth():
    """solve_ragged_host, then modes_ragged_host on GROWTH times as many trusses, each against its device entry point.
    Run in a fresh process: the ragged arena is per device and process, and earlier tests may have grown it already."""
    from tests.test_gpu_modes_ragged import device, fixture, pack

    base = [fixture(n)[1:] for n in ("bar-6", "bar-25", "bar-72")]
    rng = np.random.default_rng(5)

    def trusses(n):
        return [(j + rng.normal(0.0, 0.5, j.shape), s, c, a * (1.0 + 0.2 * rng.random(a.shape)))
                for j, s, c, a in (base[i % len(base)] for i in range(n))]

    B = 128
    p = pack(trusses(B))
    p["force"] = rng.normal(0.0, 1e3, p["xyz"].size)
    host = _lib.solve_ragged_host(3, p["joint_off"], p["member_off"], p["xyz"], p["support"], p["conn"], p["aed"], p["force"])
    dev = numpy_of(_lib.solve_ragged_device(3, device(p)))
    assert_same(host, dev, ("u", "ext", "axial", "weight", "info"))

    B *= GROWTH
    p = pack(trusses(B))
    jm = rng.random(p["support"].size)
    host = _lib.modes_ragged_host(3, p["joint_off"], p["member_off"], p["xyz"], p["support"], p["conn"], p["aed"], K,
                                  consistent=True, joint_mass=jm)
    dev = numpy_of(_lib.modes_ragged_device(3, device(p), K, consistent=True, joint_mass=cuda(jm),
                                            max_free=int(host["n_free"].max())))
    assert np.all(host["info"] == 0)
    assert_same(host, dev, ("eigval", "modes", "n_free", "info"))
    print("ragged staging ok")


def test_ragged_host_calls_share_a_growing_staging_arena():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = "from tests.test_gpu_host_staging import ragged_growth; ragged_growth()"
    res = subprocess.run([sys.executable, "-c", code], cwd=root, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "ragged staging ok" in res.stdout, res.stdout + res.stderr
