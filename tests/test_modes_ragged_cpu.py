"""Ragged modal analysis without a GPU: the exported symbols, the argument checks of tb_modes_ragged /
tb_modes_ragged_host / tb_modes_adjoint_ragged (every argument error before TB_ERR_NO_DEVICE), the Python argument
checks of autograd.modes_ragged and batch.SolveModesBatch, and the free-DOF count from the support codes."""
import ctypes as C

import numpy as np
import pytest

from oracle import truss_oracle as orc
from python_stable_3d_truss_analysis_b200 import _lib
from tests import helpers as H


def _has_cuda():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def test_symbols_exported():
    L = _lib.lib()
    for s in ("tb_modes_ragged", "tb_modes_ragged_host", "tb_modes_adjoint_ragged"):
        assert s in _lib.EXPORTS and hasattr(L, s)


def _args(dim=3, B=2, max_joint=4, max_member=5, n_modes=2, consistent=0, max_free=0):
    Bs = max(B, 1)
    keep = [np.zeros(Bs + 1, np.int64), np.zeros(Bs + 1, np.int64), np.zeros(8), np.zeros(4, np.uint8), np.zeros(10, np.int32),
            np.zeros(15), np.zeros(8), np.zeros(Bs * 20), np.zeros(Bs, np.int32)]
    jo, mo, xyz, sup, conn, aed, ev, md, info = keep
    ri = _lib.TbRaggedIn(dim, B, jo.ctypes.data, mo.ctypes.data, xyz.ctypes.data, sup.ctypes.data, conn.ctypes.data,
                         aed.ctypes.data, None, max_joint, max_member)
    mi = _lib.TbModesRaggedIn(n_modes, consistent, None, max_free)
    mo_ = _lib.TbModesRaggedOut(ev.ctypes.data, md.ctypes.data, None, info.ctypes.data)
    ai = _lib.TbModesAdjIn(ev.ctypes.data, md.ctypes.data, info.ctypes.data, ev.ctypes.data)
    ao = _lib.TbModesAdjOut(None, aed.ctypes.data, None)
    return ri, mi, mo_, ai, ao, keep


def _calls(ri, mi, mo, ai, ao):
    L = _lib.lib()
    return (L.tb_modes_ragged(C.byref(ri), C.byref(mi), C.byref(mo), None),
            L.tb_modes_ragged_host(C.byref(ri), C.byref(mi), C.byref(mo)),
            L.tb_modes_adjoint_ragged(C.byref(ri), C.byref(mi), C.byref(ai), C.byref(ao), None))


@pytest.mark.parametrize("case,want", [
    (dict(dim=4), -2),
    (dict(B=-1), -3),
    (dict(max_joint=-1), -3),
    (dict(n_modes=0), -3),
    (dict(n_modes=13), -3),                   # above the default bound d * max_joint = 12
    (dict(n_modes=5, max_free=4), -3),        # above max_free
    (dict(max_free=161), -3),
    (dict(max_free=-1), -3),
    (dict(consistent=2), -3),
    (dict(max_joint=513), -6),                # d * max_joint > 1536
    (dict(max_member=8193), -6),
])
def test_argument_errors_before_the_device(case, want):
    ri, mi, mo, ai, ao, keep = _args(**case)
    assert _calls(ri, mi, mo, ai, ao) == (want,) * 3


def test_null_arguments():
    L = _lib.lib()
    ri, mi, mo, ai, ao, keep = _args()
    assert L.tb_modes_ragged(None, C.byref(mi), C.byref(mo), None) == -1
    assert L.tb_modes_ragged(C.byref(ri), None, C.byref(mo), None) == -1
    assert L.tb_modes_ragged_host(C.byref(ri), C.byref(mi), None) == -1
    assert L.tb_modes_adjoint_ragged(C.byref(ri), C.byref(mi), None, C.byref(ao), None) == -1
    for field in ("eigval", "info"):
        bad = _lib.TbModesRaggedOut(mo.eigval, mo.modes, None, mo.info)
        setattr(bad, field, None)
        assert L.tb_modes_ragged(C.byref(ri), C.byref(mi), C.byref(bad), None) == -1
    for field in ("eigval", "modes", "info", "g_eigval"):
        bad = _lib.TbModesAdjIn(ai.eigval, ai.modes, ai.info, ai.g_eigval)
        setattr(bad, field, None)
        assert L.tb_modes_adjoint_ragged(C.byref(ri), C.byref(mi), C.byref(bad), C.byref(ao), None) == -1
    for field in ("joint_off", "member_off", "joint_xyz", "support", "conn", "member_aed"):
        bad = _lib.TbRaggedIn.from_buffer_copy(ri)
        setattr(bad, field, None)
        assert _calls(bad, mi, mo, ai, ao) == (-1,) * 3


@pytest.mark.skipif(_has_cuda(), reason="checks the no-device path")
def test_no_device():
    ri, mi, mo, ai, ao, keep = _args()
    assert _calls(ri, mi, mo, ai, ao) == (-7,) * 3
    ri.batch = 0
    assert _calls(ri, mi, mo, ai, ao) == (-7,) * 3


def test_free_dof_count_matches_every_plan():
    for name, dim, data, _ in H.shipped_cases() + H.cube7_shipped():
        joints, support, conn = orc.arrays_from_json(data, dim)[:3]
        plan = _lib.Plan(dim, conn, support)
        assert int(_lib.free_dofs_per_joint(dim, np.asarray(support, np.uint8)).sum()) == plan.n, name
    for dim in (2, 3):                                     # every code, unknown ones included
        codes = np.arange(8, dtype=np.uint8)
        want = [sum(1 for ax in range(dim) if not (c == 1 or c == 2 + ax)) for c in codes]
        assert list(_lib.free_dofs_per_joint(dim, codes)) == want


def test_python_argument_checks():
    torch = pytest.importorskip("torch")
    from python_stable_3d_truss_analysis_b200 import autograd
    from python_stable_3d_truss_analysis_b200.batch import SolveModesBatch
    from python_stable_3d_truss_analysis_b200.truss import Truss
    p = {"joint_off": torch.zeros(2, dtype=torch.int32), "member_off": torch.zeros(2, dtype=torch.int64),
         "support": torch.zeros(1, dtype=torch.uint8), "conn": torch.zeros(2, dtype=torch.int32),
         "xyz": torch.zeros(3, dtype=torch.float64), "aed": torch.zeros(3, dtype=torch.float64)}
    with pytest.raises(TypeError):                                        # joint_off must be int64
        autograd.modes_ragged(p)
    p["joint_off"] = torch.zeros(2, dtype=torch.int64)
    with pytest.raises(ValueError):
        autograd.modes_ragged(p, n_modes=0)
    with pytest.raises(TypeError):                                        # float32 coordinates
        autograd.modes_ragged(p, xyz=torch.zeros(3, dtype=torch.float32))
    with pytest.raises(ValueError):                                       # a joint_mass of the wrong size
        autograd.modes_ragged(p, joint_mass=torch.zeros(5, dtype=torch.float64))
    _, dim, data, _ = H.shipped_cases()[0]
    t = Truss(dim).LoadFromJSON(data=data)
    assert SolveModesBatch([]).size == 0
    with pytest.raises(ValueError):
        SolveModesBatch([t, Truss(5 - dim)])                              # mixed dimensions
    with pytest.raises(ValueError):
        SolveModesBatch([t], nMode=0)
    with pytest.raises(ValueError):
        SolveModesBatch([t], nMode=10 ** 4)                               # more modes than free DOFs
    with pytest.raises(ValueError):
        SolveModesBatch([t], jointMasses=[{}, {}])                        # one entry per truss
