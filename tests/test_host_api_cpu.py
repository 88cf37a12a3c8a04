"""Host-side mirror of the reference API, CPU only (nothing here launches a kernel)."""
import gzip
import json

import numpy as np
import pytest

from oracle import truss_oracle as orc
from python_stable_3d_truss_analysis_b200.generate import (AddJointNoise, GenerateRandomCubeTrusses, MoveToCentroid,
                                                             NoChange, RandomResetPin, RandomTranslation,
                                                             TrussDataAugmenterList)
from python_stable_3d_truss_analysis_b200.truss import Member, Truss
from python_stable_3d_truss_analysis_b200.type import MemberType, SupportType
from python_stable_3d_truss_analysis_b200.utils import (DimensionError, InvaildJointError, InvalidSupportTypeError,
                                                          TrussNotSolvedError, TrussNotStableError)
from tests import helpers as H


def test_types():
    assert [SupportType.NO, SupportType.PIN, SupportType.ROLLER_X, SupportType.ROLLER_Y, SupportType.ROLLER_Z] == [0, 1, 2, 3, 4]
    for name in ("NO", "PIN", "ROLLER_X", "ROLLER_Y", "ROLLER_Z"):
        assert SupportType.GetFromType(SupportType.GetFromString(name)) == name
    with pytest.raises(InvalidSupportTypeError):
        SupportType.GetFromString("WELD")
    assert SupportType.GetResistanceMask(SupportType.ROLLER_Y, 3).tolist() == [False, True, False]
    assert SupportType.GetResistanceMask(SupportType.PIN, 2).tolist() == [True, True]
    with pytest.raises(InvalidSupportTypeError):
        SupportType.GetResistanceMask(SupportType.ROLLER_Z, 2)
    assert SupportType.GetResistanceNumber(SupportType.PIN, 3) == 3
    a, b = MemberType(1, 2, 3), MemberType(1 + 1e-12, 2, 3)
    assert a == b and a.Serialize() == [1.0, 2.0, 3.0] and a.Copy() is not a
    a.Set(MemberType(4, 5, 6))
    assert a.Serialize() == [4.0, 5.0, 6.0]


def test_member_matches_oracle_element():
    m = Member((0., 0., 0.), (3., 4., 12.), 3, MemberType(2., 1e7, 0.3))
    assert m.length == 13.0 and m.k == 1e7 * 2 / 13.0
    assert np.allclose(m.matK, orc.member_matK((0., 0., 0.), (3., 4., 12.), 2., 1e7), rtol=0, atol=1e-9)
    assert m.weight == 2. * 13.0 * 0.3
    with pytest.raises(DimensionError):
        Member((0., 0.), (1., 1., 1.), 3)
    assert m.IsTension(np.array([3., 4., 12.])) and not m.IsTension(np.array([-3., -4., -12.]))


@pytest.mark.parametrize("name,dim,data,gold", H.shipped_cases(), ids=lambda v: v if isinstance(v, str) else None)
def test_json_round_trip_and_result_getters(name, dim, data, gold):
    path = f"{H.GOLDEN}/ref_data/{name.replace('_input_', '_output_')}.json"
    shipped = json.load(open(path))
    t = Truss(dim).LoadFromJSON(path, isOutputFile=True)
    assert t.isSolved and t.nJoint == len(shipped["joint"]) and t.nMember == len(shipped["member"])
    ser = t.Serialize()
    for k in ("joint", "force", "member", "displace", "external", "internal"):
        assert ser[k] == shipped[k], k
    assert abs(ser["weight"] - shipped["weight"]) <= 1e-9 * shipped["weight"]
    # packed arrays equal the oracle's reading of the same JSON
    for mine, ref in zip(t._pack(), orc.arrays_from_json(shipped, dim)):
        assert np.array_equal(np.asarray(mine), np.asarray(ref))
    # limit checks follow truss.py:429-462
    ok, vio = t.IsInternalStressAllowed(1e-3, isGetSumViolation=True)
    area = np.array([m[1][0] for m in shipped["member"]])
    want = orc.stress_violation(gold["axial"], area, 1e-3)
    assert ok == want[0] and abs(vio - want[1]) <= 1e-9 * max(1.0, abs(want[1]))
    ok, vio = t.IsDisplacementAllowed(1e-6, isGetSumViolation=True)
    want = orc.displacement_violation(gold["u"], dim, 1e-6)
    assert ok == want[0] and abs(vio - want[1]) <= 1e-9 * max(1.0, abs(want[1]))
    # resistances: external minus applied load on every supported joint (truss.py:279-291)
    res = t.GetResistances()
    sup = [j for j, (_, s) in enumerate(shipped["joint"]) if s != "NO"]
    assert sorted(res) == sup
    c = t.Copy()
    assert c.Serialize() == ser and c is not t
    stresses = t.GetInternalStresses()
    for m, f in t.GetInternalForces().items():
        assert stresses[m] == f / area[m]


def test_builders_and_errors():
    t = Truss(3)
    assert t.GetResistances() is None and t.GetInternalStresses() is None and t.GetDisplacements() is None
    for p, s in zip([(0, 0, 0), (360, 0, 0), (360, 180, 0), (0, 200, 0), (120, 100, 180)],
                    [SupportType.PIN, SupportType.ROLLER_Z, SupportType.PIN, SupportType.PIN, SupportType.NO]):
        t.AddNewJoint(p, s)
    with pytest.raises(InvaildJointError):
        t.AddExternalForce(9, (1, 0, 0))
    t.AddExternalForce(1, (0, -10000, 5000))
    t.AddExternalForce(2, (0, 0, 0))                 # dropped (truss.py:181)
    assert t.nForce == 1 and t.GetForce(1) == (0.0, -10000.0, 5000.0)
    mt = MemberType(1, 1e7, 1)
    for a, b in [(0, 4), (1, 4), (2, 4), (3, 4), (1, 2), (1, 3)]:
        t.AddNewMember(a, b, mt)
    assert (t.nJoint, t.nMember, t.nSupport, t.nResistance, t.isStable) == (5, 6, 4, 10, True)
    with pytest.raises(TrussNotSolvedError):
        t.IsInternalStressAllowed(1.0)
    t.SetMemberType(2, MemberType(9, 9, 9))
    assert t.GetMemberType(2).a == 9.0 and t.GetMemberType(1).a == 1.0     # no aliasing between members
    t.SetJointPosition(4, (100., 100., 100.))
    assert t.GetMembers()[0][2].length == (3 * 100. ** 2) ** 0.5
    t.SetSupportType(1, SupportType.PIN)
    assert t.GetSupportType(1) == SupportType.PIN and t.nResistance == 12
    assert t.GetMemberConnect(5) == (1, 3) and t.GetMemberFromConnect((1, 3)) is not None
    mask = t.GetDisplacementUnknownMask()
    assert mask.tolist() == [False] * 12 + [True] * 3
    K = t.GetKMatrix()
    assert np.array_equal(K, K.T) and K.shape == (15, 15)
    with pytest.raises(DimensionError):
        Truss(4)
    u = Truss(3)
    u.AddNewJoint((0, 0, 0), SupportType.PIN)
    u.AddNewJoint((1, 0, 0))
    u.AddNewMember(0, 1, mt)
    with pytest.raises(TrussNotStableError):
        u.Solve()


def _regen_seed42():
    return GenerateRandomCubeTrusses(gridRange=(5, 5, 5), numCubeRange=(7, 7), numEachRange=(1, 10), lengthRange=(100, 200),
                                     forceRange=[(-1000, 1000)] * 3, isDoStructuralAnalysis=False, isPrintMessage=False,
                                     seed=42)


def test_generator_reproduces_shipped_cube7_inputs():
    """generate.py:314-376 with the example.py:208-231 recipe: same `random` draw sequence -> same files."""
    mine = _regen_seed42()
    for (name, _, shipped, _), t in zip(H.cube7_shipped(), mine):
        ser = t.Serialize()
        for k in ("joint", "force", "member"):
            assert ser[k] == shipped[k], (name, k)


def test_generator_with_augmentation_matches_live_vectors():
    aug = TrussDataAugmenterList(NoChange(), MoveToCentroid(), RandomTranslation(translateRange=[-30., 30.]),
                                 AddJointNoise(noiseMeans=[0., 0., 0.], noiseStds=[10., 10., 10.]),
                                 RandomResetPin(minNumPin=5, maxNumPinRatio=0.6))
    mine = GenerateRandomCubeTrusses(gridRange=(5, 5, 5), numCubeRange=(7, 7), numEachRange=(1, 48), lengthRange=(100, 200),
                                     forceRange=[(-1000, 1000)] * 3, isDoStructuralAnalysis=False, isPrintMessage=False,
                                     seed=42, augmenter=aug)
    live = H.load_json("live_cube7_aug.json")
    assert len(mine) == len(live)
    for t, ref in zip(mine, live):
        ser = t.Serialize()
        for k in ("joint", "force", "member"):
            assert ser[k] == ref[k], k


def test_generator_other_modes_are_deterministic():
    from python_stable_3d_truss_analysis_b200.type import GenerateMethod, LinkType
    for method in (GenerateMethod.DFS, GenerateMethod.BFS, GenerateMethod.Random):
        for link in (LinkType.LeftBottom_RightTop, LinkType.RightBottom_LeftTop, LinkType.Cross, LinkType.Random):
            a = GenerateRandomCubeTrusses(gridRange=(3, 3, 3), numCubeRange=(3, 4), numEachRange=(1, 2), method=method,
                                          linkType=link, isPrintMessage=False, seed=7, isAllowParallel=(link == LinkType.Cross))
            b = GenerateRandomCubeTrusses(gridRange=(3, 3, 3), numCubeRange=(3, 4), numEachRange=(1, 2), method=method,
                                          linkType=link, isPrintMessage=False, seed=7, isAllowParallel=(link == LinkType.Cross))
            assert [t.Serialize() for t in a] == [t.Serialize() for t in b]
            assert all(t.isStable for t in a) and len(a) == 4


def test_generator_matches_live_reference_all_modes():
    with gzip.open(f"{H.GOLDEN}/live_generate_modes.json.gz", "rt") as f:
        theirs = json.load(f)
    modes = H.generator_modes()
    assert list(theirs) == [label for label, _ in modes]
    for label, kw in modes:
        assert [t.Serialize() for t in GenerateRandomCubeTrusses(**kw)] == theirs[label], label


def test_ga_trajectory_matches_live_reference_with_stub_fitness():
    """The GA operators draw from `random` exactly like ga.py:151-190: with a deterministic stand-in
    fitness (no solve) both implementations must walk the same populations."""
    from python_stable_3d_truss_analysis_b200 import ga, truss, type as types

    assert H.ga_stub_evolve(ga, truss, types) == H.load_json("live_ga_stub_bar25.json")
