"""Argument checks of tb_adjoint_ragged and of autograd.solve_ragged, without a GPU."""
import ctypes as C

import numpy as np
import pytest

from python_stable_3d_truss_analysis_b200 import _lib


def _has_cuda():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


class _Ragged:
    """Two bar trusses (3D, two joints, one member) packed back to back, as host arrays; only the pointers matter here."""

    def __init__(self, dim=3, max_joint=2, max_member=1):
        B = 2
        self.jo = np.array([0, 2, 4], np.int64)
        self.mo = np.array([0, 1, 2], np.int64)
        self.xyz = np.zeros(4 * dim)
        self.sup = np.zeros(4, np.uint8)
        self.conn = np.array([0, 1, 0, 1], np.int32)
        self.aed = np.ones(6)
        self.force = np.zeros(4 * dim)
        self.ri = _lib.TbRaggedIn(dim, B, self.jo.ctypes.data, self.mo.ctypes.data, self.xyz.ctypes.data, self.sup.ctypes.data,
                                  self.conn.ctypes.data, self.aed.ctypes.data, self.force.ctypes.data, max_joint, max_member)
        self.u = np.zeros(4 * dim)
        self.work = np.zeros(4 * dim)
        self.g_aed = np.zeros(6)
        self.info = np.zeros(B, np.int32)
        self.gi = _lib.TbAdjIn()
        self.go = _lib.TbAdjOut(None, self.g_aed.ctypes.data, None, self.info.ctypes.data)

    def call(self, ri="ri", u="u", gi="gi", go="go", work="work"):
        def ref(name, byref):
            if name is None:
                return None
            v = getattr(self, name)
            return C.byref(v) if byref else v.ctypes.data
        return _lib.lib().tb_adjoint_ragged(ref(ri, True), ref(u, False), ref(gi, True), ref(go, True), ref(work, False), None)


def test_adjoint_ragged_argument_errors():
    r = _Ragged()
    assert r.call(ri=None) == -1                                      # TB_ERR_NULL: no batch
    for name in ("u", "gi", "go", "work"):
        assert r.call(**{name: None}) == -1, name
    r.go.member_aed = None                                            # the member gradient is required
    assert r.call() == -1
    r = _Ragged()
    r.go.info = None                                                  # so is the status
    assert r.call() == -1
    r = _Ragged()
    r.ri.joint_off = None                                             # the packed arrays, as tb_solve_ragged
    assert r.call() == -1
    r = _Ragged()
    r.ri.dim = 4
    assert r.call() == -2                                             # TB_ERR_DIM
    r = _Ragged()
    r.ri.batch = -1
    assert r.call() == -3                                             # TB_ERR_SIZE
    r = _Ragged()
    r.ri.max_member = -1
    assert r.call() == -3
    r = _Ragged(max_joint=100, max_member=100)                        # d * nJ beyond the fused kernels
    assert r.call() == _lib.TB_ERR_TOO_LARGE


def test_adjoint_ragged_empty_batch_is_a_no_op():
    r = _Ragged()
    r.ri.batch = 0
    assert r.call() == 0
    assert r.call(u=None, work=None) == 0


@pytest.mark.skipif(_has_cuda(), reason="only meaningful on a machine without a GPU")
def test_adjoint_ragged_without_a_device():
    assert _Ragged().call() == _lib.TB_ERR_NO_DEVICE


def test_library_exports_tb_adjoint_ragged():
    assert "tb_adjoint_ragged" in _lib.EXPORTS
    assert hasattr(_lib.lib(), "tb_adjoint_ragged")


def _cpu_packed(torch, dim=3):
    return {"joint_off": torch.tensor([0, 2, 4]), "member_off": torch.tensor([0, 1, 2]),
            "support": torch.zeros(4, dtype=torch.uint8), "conn": torch.tensor([0, 1, 0, 1], dtype=torch.int32),
            "xyz": torch.zeros(4 * dim, dtype=torch.float64), "aed": torch.ones(6, dtype=torch.float64),
            "force": torch.zeros(4 * dim, dtype=torch.float64)}


def test_solve_ragged_rejects_bad_inputs_before_the_library():
    torch = pytest.importorskip("torch")
    from python_stable_3d_truss_analysis_b200 import autograd

    p = _cpu_packed(torch)
    with pytest.raises(TypeError, match="xyz"):
        autograd.solve_ragged(p, xyz=torch.zeros(12, dtype=torch.float32))      # wrong dtype
    with pytest.raises(ValueError, match="xyz"):
        autograd.solve_ragged(p, xyz=torch.zeros(4, 4, dtype=torch.float64))    # four columns
    with pytest.raises(ValueError, match="aed"):
        autograd.solve_ragged(p, aed=torch.ones(2, 4, dtype=torch.float64))
    with pytest.raises(ValueError, match="aed"):
        autograd.solve_ragged(p, aed=torch.ones(7, dtype=torch.float64))
    with pytest.raises(ValueError, match="force"):
        autograd.solve_ragged(p, force=torch.zeros(4, 3, dtype=torch.float64))  # loads are [d sum nJ]
    with pytest.raises(TypeError, match="force"):
        autograd.solve_ragged(p, force=np.zeros(12))                            # not a tensor
    bad = dict(p, joint_off=p["joint_off"].to(torch.int32))
    with pytest.raises(TypeError, match="joint_off"):
        autograd.solve_ragged(bad)
    with pytest.raises(TypeError, match="support"):
        autograd.solve_ragged(dict(p, support=p["support"].to(torch.int32)))
    with pytest.raises(TypeError, match="CUDA"):
        autograd.solve_ragged(p, xyz=torch.zeros(4, 3, dtype=torch.float64))    # right dtypes and shapes, on the host
