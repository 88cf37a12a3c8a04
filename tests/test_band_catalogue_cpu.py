"""The band catalogue (tests/band_catalogue.py) covers every configuration of the band kernels, read from the plans.

Coverage is read from ``plan.ts_program()["info"]`` and ``plan.info``, never from the labels, so a change to the split's
cost model or to the DOF ordering that moves a system off its target fails here instead of silently thinning the GPU
tests.  Every entry with a program is also replayed in numpy (tests/ts_replay.py) against the oracle, so that a GPU
failure on an entry can be pinned on the kernel rather than on its program.
"""
import functools

import pytest

from tests import band_catalogue as BC
from tests.test_ts_program_cpu import check


@functools.lru_cache(maxsize=None)
def summary():
    """[(entry, plan.info fields, program info or None)] for the whole catalogue."""
    out = []
    for e in BC.catalogue():
        plan = BC.plan_for(e)
        prog = plan.ts_program()
        out.append((e, {"n": plan.n, "NB16": plan.info.band_blocks}, prog["info"] if prog else None))
    return out


def _two_sided(r):
    return r[2] is not None and r[2]["nS"] > 0


def _nb(r):
    return max(r[2]["nb_top"], r[2]["nb_bottom"])


TARGETS = {f"nb={k}": (lambda r, k=k: r[2] is not None and _nb(r) == k) for k in range(1, 9)}
TARGETS.update({
    "one-sided nblk>=30": lambda r: r[2] is not None and r[2]["nS"] == 0 and r[2]["nblk"] >= 30,
    "nS=1": lambda r: _two_sided(r) and r[2]["nS"] == 1,
    "nS=8": lambda r: _two_sided(r) and r[2]["nS"] == 8,
    "nS<nb": lambda r: _two_sided(r) and r[2]["nS"] < _nb(r),
    "nS=nb": lambda r: _two_sided(r) and r[2]["nS"] == _nb(r),
    "nB=1": lambda r: _two_sided(r) and r[2]["nB"] == 1,
    "bT=1": lambda r: _two_sided(r) and r[2]["bT"] == 1,
    "nb_top!=nb_bottom": lambda r: _two_sided(r) and r[2]["nb_top"] != r[2]["nb_bottom"],
    "two-sided n%8=0": lambda r: _two_sided(r) and r[1]["n"] % 8 == 0,
    "2D": lambda r: r[2] is not None and r[0].dim == 2,
    "3D": lambda r: r[2] is not None and r[0].dim == 3,
})
TARGETS.update({f"no program NB16={k}": (lambda r, k=k: r[2] is None and r[1]["NB16"] == k) for k in range(4, 9)})


@pytest.mark.parametrize("target", list(TARGETS))
def test_catalogue_covers(target):
    hits = [r[0].label for r in summary() if TARGETS[target](r)]
    assert hits, f"no catalogue entry reaches {target}"


def test_catalogue_covers_three_nonzero_residues_of_n_mod_8():
    """Padding of the last block lands in the bottom side's first column: several residues of n mod 8, two-sided."""
    residues = {r[1]["n"] % 8 for r in summary() if _two_sided(r)}
    assert len(residues - {0}) >= 3, residues


def test_catalogue_entries_are_band_path_systems():
    """Every entry fits the band path (NB16 <= 8); labels are unique; each forced environment takes effect."""
    labels = [r[0].label for r in summary()]
    assert len(set(labels)) == len(labels)
    for e, info, ts in summary():
        assert 1 <= info["NB16"] <= 8, (e.label, info)
        if "TB_TS_SPLIT" in e.env:
            assert ts["nS"] > 0 and ts["bT"] == int(e.env["TB_TS_SPLIT"]), (e.label, ts)
        if "TB_TS_ONE_SIDED" in e.env:
            assert ts["nS"] == 0 and ts["nB"] == 0, (e.label, ts)


@pytest.mark.parametrize("region", ["top", "separator", "bottom"])
@pytest.mark.parametrize("label", ["bar-942", "t3d-10x14/split4"])
def test_failure_joints_exist(label, region):
    """The GPU failure tests zero the members of one joint whose free DOFs all lie in one region of the split."""
    e = BC.get(label)
    prog = BC.plan_for(e).ts_program()
    j = BC.joint_in(prog, e.dim, region)
    assert j is not None
    rows = BC.joint_rows(prog, e.dim)[j]
    assert rows <= BC.regions(prog)[region]
    assert len(rows) == e.dim                       # a free joint: every DOF of it is free


@pytest.mark.parametrize("label", [e.label for e in BC.catalogue()])
def test_catalogue_program_replay_matches_oracle(label):
    e = BC.get(label)
    plan = BC.plan_for(e)
    prog = plan.ts_program()
    if prog is None:
        pytest.skip("band too wide for the two-sided kernel: the 16x16 kernels take it")
    check(plan, prog, BC.arrays(e), e.dim)
