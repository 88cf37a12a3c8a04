"""Pin the oracle (oracle/truss_oracle.py) against every known-answer vector the reference ships
and against vectors produced by the live reference (SURVEY.md section 8c).  CPU only."""
import json
import os

import numpy as np
import pytest

from oracle import truss_oracle as orc
from tests import helpers as H


@pytest.mark.parametrize("name,dim,data,gold", H.shipped_cases(), ids=lambda v: v if isinstance(v, str) else None)
def test_oracle_vs_shipped_outputs(name, dim, data, gold):
    r = orc.solve(dim, *orc.arrays_from_json(data, dim))
    H.assert_close(r, gold, what=name)
    for k in H.FIELDS:
        assert H.key_sets_match(r[k], gold[k]), f"{name}: sparse key set of {k} differs above the cutoff"
    r2 = orc.solve_closed_form(dim, *orc.arrays_from_json(data, dim))
    H.assert_close(r2, gold, what=name + " (closed form)")


@pytest.mark.parametrize("name,dim,data,gold", H.cube7_shipped(), ids=lambda v: v if isinstance(v, str) else None)
def test_oracle_vs_shipped_cube7(name, dim, data, gold):
    r = orc.solve(dim, *orc.arrays_from_json(data, dim))
    H.assert_close(r, gold, what=name)


def test_oracle_vs_live_solve():
    live = H.load_json("live_solve.json")
    for name, dim, data, _ in H.shipped_cases():
        r = orc.solve(dim, *orc.arrays_from_json(data, dim))
        want = {k: np.array(v) if k != "weight" else v for k, v in live[name].items()}
        H.assert_close(r, want, tol=1e-12, what=name)


def test_oracle_vs_live_random():
    for i, case in enumerate(H.load_json("live_random.json")):
        dim = case["dim"]
        r = orc.solve(dim, *orc.arrays_from_json(case["data"], dim))
        want = {k: np.array(v) if k != "weight" else v for k, v in case["result"].items()}
        H.assert_close(r, want, tol=1e-11, what=f"random[{i}]")
        r2 = orc.solve_closed_form(dim, *orc.arrays_from_json(case["data"], dim))
        H.assert_close(r2, want, tol=1e-9, what=f"random[{i}] closed form")


def test_oracle_vs_live_cube7_aug():
    for i, gold in enumerate(H.load_json("live_cube7_aug.json")):
        r = orc.solve(3, *orc.arrays_from_json(gold, 3))
        H.assert_close(r, H.dense_from_output(gold, 3), tol=1e-11, what=f"cube7_aug[{i}]")


def test_oracle_fitness_vs_live_ga():
    g = H.load_json("live_ga_bar72.json")
    table = np.array(g["type_table"])
    blocks = [(c, v, g["allow_stress"], g["allow_displace"]) for c, v in g["cases"].items()]
    blocks.append((g["tight"]["case"], g["tight"], g["tight"]["allow_stress"], g["tight"]["allow_displace"]))
    for case, v, a_s, a_d in blocks:
        data = json.load(open(f"{H.GOLDEN}/ref_data/{case}.json"))
        joints, support, conn, _, force = orc.arrays_from_json(data, 3)
        n_bad = 0
        for gene, fit, ok_s, ok_d in list(zip(v["genes"], v["fitness"], v["stress_ok"], v["displace_ok"]))[:40]:
            f, s, d = orc.fitness(3, joints, support, conn, gene, table, force, a_s, a_d)
            assert (s, d) == (ok_s, ok_d)
            assert abs(f - fit) <= 1e-10 * abs(fit), (case, f, fit)
            n_bad += (not ok_s) or (not ok_d)
        if v is g["tight"]:
            assert n_bad > 0     # the penalty branches are exercised


def test_dof_maps_match_boolean_mask_order():
    for name, dim, data, _ in H.shipped_cases():
        _, support, *_ = orc.arrays_from_json(data, dim)
        free_idx, dof2free, sup_idx = orc.dof_maps(dim, support)
        mask = orc.free_mask(dim, support)
        assert np.array_equal(free_idx, np.nonzero(mask)[0])
        assert np.array_equal(sup_idx, np.nonzero(~mask)[0])
        assert np.array_equal(np.nonzero(dof2free >= 0)[0], free_idx)
        assert np.array_equal(dof2free[free_idx], np.arange(len(free_idx)))


def test_not_stable_rule():
    # truss.py:158-164: 3D needs >= 6 resistances and M + nRes >= 3 nJ
    joints = np.array([[0., 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1]])
    conn = np.array([[0, 3], [1, 3], [2, 3]], dtype=np.int32)
    aed = np.ones((3, 3))
    f = np.zeros(12)
    with pytest.raises(orc.NotStable):
        orc.solve(3, joints, np.array([1, 0, 0, 0], dtype=np.uint8), conn, aed, f)
    orc.solve(3, joints, np.array([1, 1, 1, 0], dtype=np.uint8), conn, aed, f)


def test_oracle_vs_live_reference_in_container():
    """The oracle against what the reference's Solve(), GetDisplacementUnknownMask() and GetKMatrix() returned
    (live_solve.json, live_kmatrix.npz; the mask and K bit for bit)."""
    live_solve = H.load_json("live_solve.json")
    kmat = np.load(os.path.join(H.GOLDEN, "live_kmatrix.npz"))
    for name, dim, data, _ in H.shipped_cases():
        joints, support, conn, aed, force = orc.arrays_from_json(data, dim)
        r = orc.solve(dim, joints, support, conn, aed, force)
        live = {k: np.array(v) if k != "weight" else v for k, v in live_solve[name].items()}
        # 1e-12, not 0: the live dicts drop entries below the 1e-10 cutoff (truss.py:358), the oracle is dense
        H.assert_close(r, live, tol=1e-12, what=name)
        free_idx, _, _ = orc.dof_maps(dim, support)
        assert np.array_equal(free_idx, kmat[name + ".free"])
        K = np.zeros((len(joints) * dim,) * 2)
        K[kmat[name + ".i"], kmat[name + ".j"]] = kmat[name + ".v"]
        assert np.array_equal(orc.assemble_K(dim, joints, conn, aed), K), name


def test_seed42_generator_inputs_reproduce_shipped():
    regen = H.load_json("live_cube7_seed42.json")
    for (name, _, shipped, _), mine in zip(H.cube7_shipped(), regen):
        for k in ("joint", "force", "member"):
            assert shipped[k] == mine[k], (name, k)
