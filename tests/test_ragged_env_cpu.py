"""Ragged batches beyond the fused kernels, without a GPU: the ordering rule the envelope kernel restates (against the
plan's own statistics), the limits of tb_solve_ragged and its argument errors, and the refusal of reverse mode."""
import ctypes as C

import numpy as np
import pytest

from oracle import truss_oracle as orc
from python_stable_3d_truss_analysis_b200 import _lib
from python_stable_3d_truss_analysis_b200.truss import Truss
from tests import helpers as H
from tests import ragged_order as RO


def _has_cuda():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def _topologies():
    out = []
    for name, dim, data, _ in H.shipped_cases():
        if name.endswith("_0") or "_input_" not in name:
            _, support, conn, _, _ = orc.arrays_from_json(data, dim)
            out.append((name, dim, support, conn))
    for i, c in enumerate(H.load_json("live_random.json")):
        _, support, conn, _, _ = orc.arrays_from_json(c["data"], c["dim"])
        out.append((f"random{i}", c["dim"], support, conn))
    for nc, seed in ((7, 1), (14, 2), (20, 3), (40, 4), (80, 5), (216, 6)):
        for k, t in enumerate(RO.host_cubes(nc, 2, seed)):
            _, support, conn, _, _ = t._pack()
            out.append((f"cube-{nc}_{k}", 3, support, conn))
    return out


TOPOLOGIES = _topologies()


@pytest.mark.parametrize("name,dim,support,conn", TOPOLOGIES, ids=[t[0] for t in TOPOLOGIES])
def test_numpy_ordering_rule_reproduces_the_plan(name, dim, support, conn):
    """The restatement the GPU tests hold the envelope kernel's order to is the plan's rule: the same envelope size,
    flops, half-bandwidth and reorder decision as tb_plan_create on the same topology."""
    plan = _lib.Plan(dim, np.asarray(conn, np.int32), np.asarray(support, np.uint8))
    want = RO.plan_order(dim, support, conn)
    info = plan.info
    assert want["reordered"] == info.reordered
    assert want["envelope_size"] == info.envelope_size
    assert want["envelope_flops"] == info.envelope_flops
    assert want["half_bandwidth"] == info.half_bandwidth
    assert sorted(want["order"]) == list(range(len(support)))


def test_shipped_cases_cover_both_reorder_decisions():
    decisions = {RO.plan_order(dim, s, c)["reordered"] for _, dim, s, c in TOPOLOGIES}
    assert decisions == {0, 1}


def test_ragged_limits():
    assert _lib.ragged_limits(3) == (512, 8192)
    assert _lib.ragged_limits(2) == (768, 8192)
    L = _lib.lib()
    a, b = C.c_int32(), C.c_int32()
    assert L.tb_ragged_limits(4, C.byref(a), C.byref(b)) == -2                  # TB_ERR_DIM
    assert L.tb_ragged_limits(3, None, C.byref(b)) == -1                        # TB_ERR_NULL
    # the generator's largest truss on a 6^3 grid and bar-942 are inside them
    prm = _lib.TbGencubeParams()
    prm.grid[:] = (6, 6, 6)
    prm.ncube_lo = prm.ncube_hi = 216
    prm.link_type, prm.n_type, prm.max_attempts = 2, 1, 1
    mj, mm, mc = C.c_int32(), C.c_int32(), C.c_int32()
    assert L.tb_gencube_limits(C.byref(prm), C.byref(mj), C.byref(mm), C.byref(mc)) == 0
    assert (mj.value, mm.value) == (343, 5184)
    assert mj.value <= 512 and mm.value <= 8192
    # the fused launch of a routed batch is sized at the routing limits: it must fit k_dense16 (hence the fused kernels)
    assert _lib.small_path_fits(3, 48, 192) and _lib.small_path_fits(2, 72, 224)
    assert _lib.small_path_fits(3, 32, 119)                                     # cube-7 is under them


class _Batch:
    """Two trusses packed back to back as host arrays (only the pointers and sizes matter here)."""

    def __init__(self, dim=3, max_joint=2, max_member=1):
        self.jo = np.array([0, 2, 4], np.int64)
        self.mo = np.array([0, 1, 2], np.int64)
        self.xyz = np.zeros(4 * dim)
        self.sup = np.zeros(4, np.uint8)
        self.conn = np.array([0, 1, 0, 1], np.int32)
        self.aed = np.ones(6)
        self.force = np.zeros(4 * dim)
        self.ri = _lib.TbRaggedIn(dim, 2, self.jo.ctypes.data, self.mo.ctypes.data, self.xyz.ctypes.data, self.sup.ctypes.data,
                                  self.conn.ctypes.data, self.aed.ctypes.data, self.force.ctypes.data, max_joint, max_member)
        self.u = np.zeros(4 * dim)
        self.info = np.zeros(2, np.int32)
        self.order = np.zeros(4, np.int32)
        self.env = np.zeros(2, np.int64)
        self.bo = _lib.TbBatchOut(self.u.ctypes.data, None, None, None, self.info.ctypes.data)

    def calls(self):
        L = _lib.lib()
        return {"device": L.tb_solve_ragged(C.byref(self.ri), C.byref(self.bo), None),
                "host": L.tb_solve_ragged_host(C.byref(self.ri), C.byref(self.bo)),
                "env": L.tb_solve_ragged_env(C.byref(self.ri), C.byref(self.bo), None),
                "order": L.tb_ragged_env_order(C.byref(self.ri), self.order.ctypes.data, self.env.ctypes.data, None)}


def test_argument_errors_beyond_the_new_limits():
    for dim, mj in ((3, 513), (2, 769)):
        r = _Batch(dim=dim, max_joint=mj, max_member=10)
        assert set(r.calls().values()) == {_lib.TB_ERR_TOO_LARGE}, dim
    r = _Batch(max_joint=100, max_member=8193)
    assert set(r.calls().values()) == {_lib.TB_ERR_TOO_LARGE}
    r = _Batch()
    r.ri.dim = 4
    assert set(r.calls().values()) == {-2}
    r = _Batch()
    r.ri.max_member = -1
    assert set(r.calls().values()) == {-3}
    r = _Batch()
    r.ri.conn = None
    assert set(r.calls().values()) == {-1}
    r = _Batch()
    L = _lib.lib()
    assert L.tb_solve_ragged(C.byref(r.ri), None, None) == -1
    assert L.tb_solve_ragged_env(C.byref(r.ri), None, None) == -1
    assert L.tb_ragged_env_order(C.byref(r.ri), None, r.env.ctypes.data, None) == -1
    assert L.tb_ragged_env_order(C.byref(r.ri), r.order.ctypes.data, None, None) == -1
    r.ri.batch = 0                                                              # not an argument error (a no-op with a GPU)
    assert set(r.calls().values()) <= {0, _lib.TB_ERR_NO_DEVICE}


def test_compact_layout_is_still_refused():
    r = _Batch(max_joint=300, max_member=1000)                                 # a batch for the envelope kernel
    uf = np.zeros(8)
    bo = _lib.TbBatchOut(None, None, None, None, None, uf.ctypes.data, None)
    L = _lib.lib()
    assert L.tb_solve_ragged(C.byref(r.ri), C.byref(bo), None) == -3
    assert L.tb_solve_ragged_host(C.byref(r.ri), C.byref(bo)) == -3
    assert L.tb_solve_ragged_env(C.byref(r.ri), C.byref(bo), None) == -3


@pytest.mark.skipif(_has_cuda(), reason="only meaningful on a machine without a GPU")
def test_admitted_large_batch_without_a_device():
    """A batch the fused kernels refuse but the envelope kernel admits gets as far as the device check."""
    assert not _lib.small_path_fits(3, 300, 1000)
    r = _Batch(max_joint=300, max_member=1000)
    assert set(r.calls().values()) == {_lib.TB_ERR_NO_DEVICE}
    with pytest.raises(_lib.TrussLibError) as ei:                               # PackedDataset.solve's entry
        _lib.solve_ragged_host(3, r.jo, r.mo, r.xyz, r.sup, r.conn, r.aed, r.force)
    assert ei.value.code == _lib.TB_ERR_NO_DEVICE


def test_autograd_refuses_a_large_batch_before_any_launch():
    torch = pytest.importorskip("torch")
    from python_stable_3d_truss_analysis_b200 import autograd

    p = {"joint_off": torch.tensor([0, 2, 4]), "member_off": torch.tensor([0, 1, 2]),
         "support": torch.zeros(4, dtype=torch.uint8), "conn": torch.tensor([0, 1, 0, 1], dtype=torch.int32),
         "xyz": torch.zeros(12, dtype=torch.float64), "aed": torch.ones(6, dtype=torch.float64),
         "force": torch.zeros(12, dtype=torch.float64)}
    # (host tensors: a launch would be refused for them as well, so the refusal must come before the tensors are used)
    if _has_cuda():
        p = {k: v.cuda() for k, v in p.items()}
    with pytest.raises(_lib.TrussLibError) as ei:
        autograd.solve_ragged(p, max_joint=300, max_member=1000)
    assert ei.value.code == _lib.TB_ERR_TOO_LARGE


def test_library_exports_the_envelope_entry_points():
    for s in ("tb_solve_ragged_env", "tb_ragged_env_order", "tb_ragged_limits"):
        assert s in _lib.EXPORTS and hasattr(_lib.lib(), s)
    assert "tb_ragenv.cu" in _lib.SOURCES


def test_truss_views_of_generated_cubes_are_solvable_topologies():
    """(the host-generated cubes above are what the GPU tests solve: the counting rule holds for them)"""
    for t in RO.host_cubes(40, 2, 4):
        xyz, sup, conn, _, _ = t._pack()
        assert orc.is_stable(3, sup, len(conn))
        assert isinstance(t, Truss)
