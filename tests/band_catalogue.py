"""A catalogue of band-path systems that together reach every configuration the band kernels can be given.

``k_band_ts`` (csrc/tb_bandts.cu) is instantiated per nb = max(nb_top, nb_bottom) (1 .. 8), runs a one-sided program or
a top / separator / bottom split chosen by a cost model (csrc/tb_tsplan.cu), and pads the last block of the top side
(the bottom side's first column when n % 8 != 0).  Systems whose band is too wide for the 8x8 program run on the 16x16
kernels k_band1/2/3 (csrc/tb_band.cu).  Each entry is ``(label, dim, data, env)``: a truss in the reference's JSON form
and the environment under which its plan is built (``{}``, ``{"TB_TS_SPLIT": k}`` or ``{"TB_TS_ONE_SIDED": "1"}``;
both are read when the plan builds its program, nowhere else).  tests/test_band_catalogue_cpu.py checks, from the plans
themselves, that the catalogue covers every configuration; tests/test_gpu_band_kernels.py runs it on the GPU.
"""
from __future__ import annotations

import functools
import json
import os
from typing import NamedTuple

import numpy as np

from oracle import truss_oracle as orc
from python_stable_3d_truss_analysis_b200 import _lib
from tests import helpers as H


class Entry(NamedTuple):
    label: str
    dim: int
    data: dict
    env: dict


def _shipped(name):
    return json.load(open(os.path.join(H.GOLDEN, "ref_data", f"{name}_input_0.json")))


def _tower(dim, per_level, levels):
    return H.tower(dim, per_level, levels, seed=per_level)


@functools.lru_cache(maxsize=None)
def catalogue():
    """The entries.  Labels of the same system differ only after the '/': the part before it names the truss."""
    b942 = _shipped("bar-942")
    t2_4 = _tower(2, 4, 40)
    t3_10 = _tower(3, 10, 14)
    out = [
        # the automatic split, nb = 1 .. 8
        ("t2d-4x40", 2, t2_4, {}),                          # nb 1, nS = nb = 1, n % 8 = 0
        ("t2d-6x30", 2, _tower(2, 6, 30), {}),              # nb 2, nS = nb = 2, n % 8 = 4
        ("t3d-3x30", 3, _tower(3, 3, 30), {}),              # nb 3, n % 8 = 5
        ("t3d-5x24", 3, _tower(3, 5, 24), {}),              # nb 4, n % 8 = 1
        ("t3d-8x16", 3, _tower(3, 8, 16), {}),              # nb 5
        ("t3d-7x18", 3, _tower(3, 7, 18), {}),              # nb 6
        ("t3d-9x14", 3, _tower(3, 9, 14), {}),              # nb 7, n % 8 = 7
        ("t3d-10x14", 3, t3_10, {}),                        # nb 8, n % 8 = 6
        ("bar-942", 3, b942, {}),                           # the benchmark truss: nb 7, nS 5
        ("bar-120", 3, _shipped("bar-120"), {}),            # nb_top 7, nb_bottom 6, nS 6 of 14 block columns
        # forced splits and one-sided programs
        ("t3d-10x14/split4", 3, t3_10, {"TB_TS_SPLIT": "4"}),          # nS = 8, the maximum
        ("t2d-4x40/split37", 2, t2_4, {"TB_TS_SPLIT": "37"}),          # nB = 1
        ("t2d-4x40/split1", 2, t2_4, {"TB_TS_SPLIT": "1"}),            # bT = 1
        ("bar-942/split81", 3, b942, {"TB_TS_SPLIT": "81"}),           # nB = 1, nb_top 7 != nb_bottom 5
        ("t2d-4x40/one-sided", 2, t2_4, {"TB_TS_ONE_SIDED": "1"}),     # 39 block columns on one warp
        ("t3d-10x14/one-sided", 3, t3_10, {"TB_TS_ONE_SIDED": "1"}),   # 49 block columns, nb 8
        # bands too wide for the 8x8 program: the 16x16 kernels, NB16 = 4 .. 8
        ("t3d-11x12", 3, _tower(3, 11, 12), {}),
        ("t3d-13x10", 3, _tower(3, 13, 10), {}),
        ("t3d-15x9", 3, _tower(3, 15, 9), {}),
        ("t3d-19x8", 3, _tower(3, 19, 8), {}),
        ("t3d-21x7", 3, _tower(3, 21, 7), {}),
    ]
    return [Entry(*e) for e in out]


def get(label):
    return next(e for e in catalogue() if e.label == label)


def arrays(entry):
    """(joints, support, conn, aed, force) of the entry's truss, as the oracle takes them."""
    return orc.arrays_from_json(entry.data, entry.dim)


def plan_for(entry):
    """The entry's plan, with its environment set only while the plan (and so its band program) is built."""
    joints, support, conn, aed, force = arrays(entry)
    old = {k: os.environ.get(k) for k in entry.env}
    os.environ.update(entry.env)
    try:
        return _lib.Plan(entry.dim, conn, support)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def ts_nb(prog):
    """The k_band_ts instantiation a program runs on: max(nb_top, nb_bottom)."""
    return max(prog["info"]["nb_top"], prog["info"]["nb_bottom"])


def inputs(plan, entry, B, seed=0):
    """B systems of the entry's topology, each with its own member areas and load vector: (xyz [nJ, d] shared,
    aed [B, M, 3], force [B, N])."""
    joints, support, conn, aed, force = arrays(entry)
    rng = np.random.default_rng(seed)
    aedb = np.repeat(aed[None], B, axis=0)
    aedb[:, :, 0] *= rng.uniform(0.5, 2.0, size=(B, plan.M))
    F = force.reshape(1, -1) * rng.uniform(0.5, 2.0, size=(B, 1)) + rng.uniform(-1.0, 1.0, size=(B, plan.N))
    return np.ascontiguousarray(joints), aedb, F


def regions(prog):
    """The plan-order rows of the top side's own columns, of the separator and of the bottom side's own columns, read
    from the program's row maps (rownat: the plan-order row of each program row, -1 on padding)."""
    info = prog["info"]
    top, bot = prog["side"]
    own_top = top["rownat"][:8 * info["bT"]]
    sep = top["rownat"][8 * info["bT"]:8 * (info["bT"] + info["nS"])]
    own_bot = bot["rownat"][:8 * info["nB"]]
    return {"top": set(own_top[own_top >= 0].tolist()), "separator": set(sep[sep >= 0].tolist()),
            "bottom": set(own_bot[own_bot >= 0].tolist())}


def joint_rows(prog, dim):
    """{free joint: plan-order rows of its free DOFs}, from the program's rowdof / rownat maps."""
    out = {}
    top = prog["side"][0]
    nat, dof = top["rownat"], top["rowdof"]
    for r, d in zip(nat.tolist(), dof.tolist()):
        if r >= 0:
            out.setdefault(d // dim, set()).add(r)
    bot = prog["side"][1]
    for r, d in zip(bot["rownat"].tolist(), bot["rowdof"].tolist()):
        if r >= 0:
            out.setdefault(d // dim, set()).add(r)
    return out


def joint_in(prog, dim, region):
    """A free joint whose free DOFs all lie in one region ("top", "separator", "bottom"), or None: of all such joints the
    middle one in the elimination order of the side that owns the region, so that good columns come before and after it."""
    reg = regions(prog)[region]
    cand = sorted(((min(rows) if region != "bottom" else -max(rows)), j)
                  for j, rows in joint_rows(prog, dim).items() if rows <= reg)
    return cand[len(cand) // 2][1] if cand else None
