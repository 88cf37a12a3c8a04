"""The band kernels on the GPU over the band catalogue (tests/band_catalogue.py): every instantiation k_band_ts<1..8>,
forced splits (nS = 8, a one-column bottom side, bT = 1), long one-sided programs, padded last blocks, the grid-stride
loop with several systems per CTA, pivot failures confined to one part of the split, the adjoint, and the two-stream
half-batch path of the 16x16 kernels.

Every test records the CUDA kernels of its call with torch.profiler and asserts that the kernel it targets ran, so no
test can pass on a different kernel than the one it names.  Batch-size tests call Plan.solve_device: the blocking host
entry point would cut a batch into chunks."""
import numpy as np
import pytest

from oracle import truss_oracle as orc
from tests import band_catalogue as BC
from tests import helpers as H
from tests.test_gpu_adjoint import assert_grads_close, device_adjoint, oracle_grads, random_grads

pytestmark = pytest.mark.gpu

OUTS = ("u", "ext", "axial", "weight", "info")
BE_TOL = 1e-14          # backward error of a binary64 Cholesky solve is ~1e-16 (measured on the numpy replay: <= 1.1e-16)
PROGRAM_LABELS = [e.label for e in BC.catalogue() if BC.plan_for(e).ts_program() is not None]


def _torch():
    import torch
    return torch


def n_sm():
    return _torch().cuda.get_device_properties(0).multi_processor_count


def many_per_cta():
    """A batch size at which every CTA of k_band_ts (at most seven per SM) runs at least two systems."""
    return 2 * 7 * n_sm() + 3


def band_plan(label):
    e = BC.get(label)
    plan = BC.plan_for(e)
    prog = plan.ts_program()
    plan.set_path(2)
    return e, plan, prog


def assert_vs_oracle(e, aed, F, out, b, what):
    joints, support, conn, _, _ = BC.arrays(e)
    want = orc.solve(e.dim, joints, support, conn, aed[b], F[b])
    H.assert_close({k: out[k][b] for k in H.FIELDS} | {"weight": out["weight"][b]}, want, what=f"{what}[{b}]")
    be = H.backward_error(e.dim, joints, support, conn, aed[b], F[b], out["u"][b])
    assert be <= BE_TOL, f"{what}[{b}]: backward error {be:.2e}"


# --------------------------------------------------------------------------- oracle parity over the catalogue
@pytest.mark.parametrize("label", PROGRAM_LABELS)
def test_band_ts_vs_oracle(label):
    """Five systems with their own member areas and loads through k_band_ts<nb>, against the oracle (1e-9 per field)
    and with a backward error at rounding level."""
    e, plan, prog = band_plan(label)
    B = 5
    xyz, aed, F = BC.inputs(plan, e, B, seed=3)
    out, seen = H.cuda_kernels(lambda: H.solve_device_np(plan, B, xyz, aed, F))
    print(f"{label}: {seen}")
    assert H.band_kernels(seen) == [f"k_band_ts<{BC.ts_nb(prog)}>"], seen
    assert not out["info"].any(), out["info"]
    for b in range(B):
        assert_vs_oracle(e, aed, F, out, b, label)


# --------------------------------------------------------------------------- the grid-stride loop
def batch_and_solo(label, zero_joints=None, seed=5):
    """many_per_cta() systems of an entry solved as one batch (twice) and each on its own (B = 1).  zero_joints maps a
    batch position to joints whose members all get E = 0 there.  Returns (entry, program, inputs, batch, second batch,
    solo, kernel tags of the first batch)."""
    torch = _torch()
    e, plan, prog = band_plan(label)
    B = many_per_cta()
    xyz, aed, F = BC.inputs(plan, e, B, seed=seed)
    conn = BC.arrays(e)[2]
    for b, joints in (zero_joints or {}).items():
        for j in joints:
            aed[b, (conn == j).any(axis=1), 1] = 0.0
    out, seen = H.cuda_kernels(lambda: H.solve_device_np(plan, B, xyz, aed, F))
    again = H.solve_device_np(plan, B, xyz, aed, F)
    dev = torch.device("cuda:0")
    td = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    x_t, a_t, f_t = td(xyz), td(aed), td(F)
    f64 = dict(dtype=torch.float64, device=dev)
    solo = {"u": torch.empty(B, plan.N, **f64), "ext": torch.empty(B, plan.N, **f64), "axial": torch.empty(B, plan.M, **f64),
            "weight": torch.empty(B, **f64), "info": torch.empty(B, dtype=torch.int32, device=dev)}
    for b in range(B):
        plan.solve_device(1, x_t, f_t[b:b + 1], aed=a_t[b:b + 1], out={k: v[b:b + 1] for k, v in solo.items()})
    torch.cuda.synchronize()
    solo = {k: v.cpu().numpy() for k, v in solo.items()}
    return e, prog, (xyz, aed, F), out, again, solo, seen


@pytest.mark.parametrize("label", ["t2d-4x40", "t3d-10x14", "t3d-10x14/one-sided"])
def test_band_ts_batch_equals_single_solves(label):
    """2 * 7 * SMs + 3 systems: every CTA runs at least two systems in its grid-stride loop, and each system's results
    are bit for bit those of the same system solved alone."""
    e, prog, (xyz, aed, F), out, again, solo, seen = batch_and_solo(label)
    print(f"{label}: {seen}")
    assert H.band_kernels(seen) == [f"k_band_ts<{BC.ts_nb(prog)}>"], seen
    assert not out["info"].any()
    for k in OUTS:
        assert np.array_equal(out[k], solo[k]), k
        assert np.array_equal(out[k], again[k]), k
    for b in (0, len(F) - 1):
        assert_vs_oracle(e, aed, F, out, b, label)


@pytest.mark.parametrize("label", ["bar-942", "t3d-10x14/split4"])
def test_band_ts_failures_are_local(label):
    """A free joint whose members all have E = 0 makes its rows of K_ff zero: the first of its pivots the owning side
    meets is 0.  One system fails in the top side's own columns, one in the separator, one in the bottom side's own
    columns and one on both sides, among good systems that share their CTAs.  info - 1 is the plan-order row of one
    of the failing joint's DOFs; when both sides fail, the bottom side's row is reported (DESIGN.md section 3); the
    failing outputs are zeros, everything is bit for bit the solo solves, and info does not change on a second call."""
    e, plan, prog = band_plan(label)
    jt, js, jb = (BC.joint_in(prog, e.dim, r) for r in ("top", "separator", "bottom"))
    rows = BC.joint_rows(prog, e.dim)
    B = many_per_cta()
    expect = {0: jt, 1: js, 2: jb, B - 1: jb}
    zero = {0: [jt], 1: [js], 2: [jb], B - 1: [jt, jb]}
    e, prog, (xyz, aed, F), out, again, solo, seen = batch_and_solo(label, zero_joints=zero)
    print(f"{label}: {seen}; info {[int(out['info'][b]) for b in sorted(expect)]}")
    assert H.band_kernels(seen) == [f"k_band_ts<{BC.ts_nb(prog)}>"], seen
    for b, j in expect.items():
        assert out["info"][b] > 0 and out["info"][b] - 1 in rows[j], (b, int(out["info"][b]), sorted(rows[j]))
        for k in ("u", "ext", "axial", "weight"):
            assert not np.any(out[k][b]), (b, k)
    good = np.setdiff1d(np.arange(B), list(expect))
    assert not out["info"][good].any()
    for k in OUTS:
        assert np.array_equal(out[k], solo[k]), k
        assert np.array_equal(out[k], again[k]), k
    for b in (3, B - 2):
        assert_vs_oracle(e, aed, F, out, b, label)


# --------------------------------------------------------------------------- reverse mode
@pytest.mark.parametrize("label", ["t3d-10x14", "bar-942/split81"])
def test_band_ts_adjoint_vs_oracle(label):
    e, plan, prog = band_plan(label)
    joints, support, conn, _, _ = BC.arrays(e)
    B = 2
    xyz, aed, F = BC.inputs(plan, e, B, seed=9)
    grads = random_grads(np.random.default_rng(9), B, plan.N, plan.M)
    (fwd, got), seen = H.cuda_kernels(lambda: device_adjoint(plan, joints, aed, F, grads))
    print(f"{label}: {seen}")
    assert H.band_kernels(seen) == [f"k_band_ts<{BC.ts_nb(prog)}>"], seen
    assert not fwd["info"].any() and not got["info"].any()
    for b in range(B):
        assert_grads_close(got, oracle_grads(e.dim, joints, support, conn, aed[b], F[b], grads, b), b, what=label)


# --------------------------------------------------------------------------- the two-stream half-batch path
def test_half_batch_two_streams(tmp_path):
    """NB16 4 without a two-sided program at 7 * SMs systems: two half-batches on two streams (two k_prep launches),
    bit for bit the unsplit batch (TB_LARGE_SPLIT=0) and a 32-system batch around the split point at 4 * SMs."""
    label = "t3d-11x12"
    e, plan, prog = band_plan(label)
    assert prog is None and plan.info.band_blocks == 4
    B, n0 = 7 * n_sm(), 4 * n_sm()
    xyz, aed, F = BC.inputs(plan, e, B, seed=13)
    split, seen = H.cuda_kernels(lambda: H.solve_device_np(plan, B, xyz, aed, F))
    print(f"split: {seen}")
    assert seen.get("k_prep<3>") == 2 and H.band_kernels(seen) == ["k_band2<4>"], seen
    assert not split["info"].any()
    lo, hi = n0 - 16, n0 + 16
    part, seen_p = H.cuda_kernels(lambda: H.solve_device_np(plan, hi - lo, xyz, aed[lo:hi], F[lo:hi]))
    assert seen_p.get("k_prep<3>") == 1, seen_p
    (whole, seen_w), = H.run_band_child(tmp_path, {"TB_LARGE_SPLIT": "0"}, [{"label": label, "B": B, "seed": 13}])
    print(f"unsplit: {seen_w}")
    assert seen_w.get("k_prep<3>") == 1 and len(H.band_kernels(seen_w)) == 1, seen_w
    for k in OUTS:
        assert np.array_equal(split[k], whole[k]), k
        assert np.array_equal(split[k][lo:hi], part[k]), k
    for b in (0, n0 - 1, n0, B - 1):
        assert_vs_oracle(e, aed, F, split, b, label)
