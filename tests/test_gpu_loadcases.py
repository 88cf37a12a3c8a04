"""Load cases of one truss on the GPU (tb_solve_loadcases / tb_solve_loadcases_host, shared_factor=True): on the band
path the truss is assembled (k_prep) and factorised (k_band3 / k_band1) once, for load case 0, and every load case then
runs only the two triangular substitutions against that factor, in one of two kernels (csrc/tb_band.cu):

  k_band_subst8<NB>      eight load cases per warp on the FP64 tensor cores; y of the whole system stays in shared
                         memory, so it runs while (2 (NB+1) 256 + (NB+1) 128 + 128 + nb16 128) 8 bytes <= 200 KB; its grid
                         is capped at SMs * floor(220 KB / (that + 1 KB)) tiles and grid-strides beyond;
  k_band_subst<NB, 4>    one warp per load case, four per CTA: longer systems, or any system under TB_SUBST_TILE=1.

The systems: every truss of the band catalogue (NB16 = 1 .. 8, 2D and 3D, zero-skipped and full sub-diagonal blocks), a
tower with n % 16 = 0, the shipped fixtures forced onto the band path (nb16 = 1 .. 7, nb16 <= NB on bar-6 and bar-10) and a
long 2D ladder that takes the warp-per-load-case kernel by itself.  Every call records its CUDA kernels, so no test passes
on a kernel other than the one it names; results are checked against a dense numpy solve (1e-9 norm-wise per field) and
by their backward error, which a Cholesky solve in binary64 keeps at rounding level whatever the conditioning."""
import functools
import json
import os

import numpy as np
import pytest

from oracle import truss_oracle as orc
from python_stable_3d_truss_analysis_b200 import _lib
from tests import band_catalogue as BC
from tests import helpers as H
from tests.test_gpu_adjoint import FIELDS as GRAD_FIELDS
from tests.test_gpu_adjoint import assert_grads_close, device_adjoint, oracle_grads, random_grads

pytestmark = pytest.mark.gpu

OUTS = ("u", "ext", "axial", "weight", "info")
BE_TOL = 1e-14          # backward error of a binary64 Cholesky solve is ~1e-16
BATCHES = (1, 2, 7, 8, 9, 17)   # one case, partial tiles, an exact tile, a tile boundary; a partial last CTA of four
NB_CASES = max(BATCHES)


def _torch():
    import torch
    return torch


def n_sm():
    return _torch().cuda.get_device_properties(0).multi_processor_count


def ladder():
    """A 2D ladder of 790 levels (tower(2, 2, 790)) pinned at the bottom, at the top and every 40 levels: n = 3076, 193
    block columns, so y does not fit k_band_subst8's shared memory (204 KB) and the warp-per-load-case kernel runs; the
    member products (95 KB) still fit k_prep.  The intermediate supports keep cond(K_ff) near 1e5 (1e10 without them)."""
    data = H.tower(2, 2, 790, seed=2)
    for i, j in enumerate(data["joint"]):
        if (i // 2) % 40 == 0 or i // 2 == 789:
            j[1] = "PIN"
    return data


@functools.lru_cache(maxsize=None)
def systems():
    out = {e.label: (e.dim, e.data) for e in BC.catalogue() if "/" not in e.label}
    out["t2d-4x41"] = (2, H.tower(2, 4, 41, seed=4))                 # n = 320: no padded last block
    for name in ("bar-6", "bar-10", "bar-25", "bar-72"):              # (bar-120 is in the catalogue)
        out[name] = (H.dim_of(name + "_"), json.load(open(os.path.join(H.GOLDEN, "ref_data", f"{name}_input_0.json"))))
    out["ladder"] = (2, ladder())
    return out


LABELS = list(systems())


class System:
    """A truss on the band path with its dense K, the launch parameters of the substitution kernels, and a reference
    solve of any number of load cases (one dense factorisation of K_ff for all of them)."""

    def __init__(self, label, dim=None, data=None, dense=True):
        self.label = label
        self.dim, self.data = (dim, data) if data is not None else systems()[label]
        self.joints, self.support, self.conn, self.aed, self.force = orc.arrays_from_json(self.data, self.dim)
        self.plan = _lib.Plan(self.dim, self.conn, self.support)
        self.plan.set_path(2)
        self.N, self.M, self.n = self.plan.N, self.plan.M, self.plan.n
        self.NB = self.plan.info.band_blocks
        self.nb16 = max(1, (self.n + 15) // 16)
        self.smem8 = (2 * (self.NB + 1) * 256 + (self.NB + 1) * 128 + 128 + self.nb16 * 128) * 8
        self.subst = f"k_band_subst8<{self.NB}>" if self.smem8 <= 200 * 1024 else f"k_band_subst<{self.NB}>"
        self.factor = f"k_band3<{self.NB}>" if self.NB <= 5 else f"k_band1<{self.NB}>"
        self.mask = orc.free_mask(self.dim, self.support)
        if dense:                              # (the oracle has no K for a zero-length member)
            self.K = orc.assemble_K(self.dim, self.joints, self.conn, self.aed)
            self.Kff = self.K[self.mask][:, self.mask]

    def loads(self, B, seed=1):
        rng = np.random.default_rng(seed)
        return self.force.reshape(1, -1) * rng.uniform(0.5, 2.0, size=(B, 1)) + rng.uniform(-1.0, 1.0, size=(B, self.N))

    def solve(self, F, **kw):
        return H.solve_device_np(self.plan, F.shape[0], self.joints, self.aed, F, shared_factor=True, **kw)

    def reference(self, F):
        """orc.solve for every row of F, with one factorisation of K_ff (the closed-form axial forces of
        orc.solve_closed_form)."""
        B, d = F.shape[0], self.dim
        U = np.zeros_like(F)
        U[:, self.mask] = np.linalg.solve(self.Kff, F[:, self.mask].T).T
        ext = F.copy()
        ext[:, ~self.mask] = U @ self.K[~self.mask].T
        dx = self.joints[self.conn[:, 1]] - self.joints[self.conn[:, 0]]
        L = np.sqrt((dx ** 2).sum(axis=1))
        Uj = U.reshape(B, -1, d)
        du = Uj[:, self.conn[:, 1]] - Uj[:, self.conn[:, 0]]
        axial = self.aed[:, 1] * self.aed[:, 0] / L * (du * (dx / L[:, None])).sum(axis=2)
        return {"u": U, "ext": ext, "axial": axial, "weight": orc.weight(self.joints, self.conn, self.aed)}

    def backward_errors(self, F, U):
        """H.backward_error of every row, on the K_ff assembled once."""
        uf, ff = U[:, self.mask], F[:, self.mask]
        r = np.abs(uf @ self.Kff.T - ff).max(axis=1)
        return r / (np.abs(self.Kff).sum(axis=1).max() * np.abs(uf).max(axis=1) + np.abs(ff).max(axis=1))

    def check(self, out, F, want, what):
        assert not out["info"].any(), (what, out["info"])
        for b in range(F.shape[0]):
            H.assert_close({k: out[k][b] for k in H.FIELDS} | {"weight": out["weight"][b]},
                           {k: want[k][b] for k in H.FIELDS} | {"weight": want["weight"]}, what=f"{what}[{b}]")
        be = self.backward_errors(F, out["u"])
        assert be.max() <= BE_TOL, f"{what}: backward error {be.max():.2e} at load case {int(be.argmax())}"


@functools.lru_cache(maxsize=None)
def system(label):
    return System(label)


@functools.lru_cache(maxsize=None)
def reference_cases(label):
    s = system(label)
    F = s.loads(NB_CASES)
    want = s.reference(F)
    one = orc.solve(s.dim, s.joints, s.support, s.conn, s.aed, F[0])            # the oracle itself, on one load case
    H.assert_close({k: want[k][0] for k in H.FIELDS} | {"weight": want["weight"]}, one, what=f"{label} reference")
    return F, want


@functools.lru_cache(maxsize=None)
def default_runs(label):
    """{B: (outputs, kernel tags)} of the first B load cases, for every B of BATCHES."""
    s = system(label)
    F, _ = reference_cases(label)
    return {B: H.cuda_kernels(lambda: s.solve(F[:B])) for B in BATCHES}


def assert_same(a, b, what, keys=OUTS):
    for k in keys:
        assert np.array_equal(a[k], b[k]), (what, k)


# --------------------------------------------------------------------------- routing and parity
@pytest.mark.parametrize("label", LABELS)
def test_shared_factor_routing_and_parity(label):
    """One k_prep, one factorisation (k_band3<NB> for NB <= 5, k_band1<NB> beyond, never k_band_ts) and one
    substitution launch (k_band_subst8<NB>, or k_band_subst<NB> on the ladder) at every batch size, the one-case batch
    included; every load case against the reference and at a backward error of rounding level; a load case's bits do not
    depend on the batch size."""
    s = system(label)
    F, want = reference_cases(label)
    runs = default_runs(label)
    print(f"{label} (NB {s.NB}, nb16 {s.nb16}, smem8 {s.smem8 // 1024} KB): {runs[NB_CASES][1]}")
    for B, (out, seen) in runs.items():
        assert seen.get(f"k_prep<{s.dim}>") == 1, (B, seen)
        assert H.band_kernels(seen) == [s.factor] and seen[s.factor] == 1, (B, seen)
        assert H.subst_kernels(seen) == [s.subst] and seen[s.subst] == 1, (B, seen)
        s.check(out, F[:B], {k: v[:B] for k, v in want.items() if k != "weight"} | {"weight": want["weight"]}, f"{label} B={B}")
        assert_same(out, {k: v[:B] for k, v in runs[NB_CASES][0].items()}, f"{label} B={B}")


@pytest.mark.parametrize("name,path", [("bar-72", 0), ("bar-72", 1), ("bar-942", 1)])
def test_shared_factor_is_ignored_off_the_band_path(name, path):
    """The fused and tiled pipelines factorise every system: shared_factor changes nothing, bit for bit."""
    s = System(name, 3, json.load(open(os.path.join(H.GOLDEN, "ref_data", f"{name}_input_0.json"))))
    s.plan.set_path(path)
    F = s.loads(9)
    shared = s.solve(F)
    indep = H.solve_device_np(s.plan, 9, s.joints, s.aed, F)
    assert not indep["info"].any()
    assert_same(shared, indep, f"{name} path {path}")


@pytest.fixture(scope="module")
def tile1_runs(tmp_path_factory):
    """Under TB_SUBST_TILE=1 (read once per process: a child process): every system at every batch size, and the
    failing trusses of test_shared_factor_failures at 13 load cases."""
    tmp = tmp_path_factory.mktemp("subst_tile1")
    jobs = []
    for label in LABELS:
        s = system(label)
        F, _ = reference_cases(label)
        path = str(tmp / f"{label}.npy")
        np.save(path, F)
        jobs += [{"label": label, "dim": s.dim, "data": s.data, "B": B, "seed": 0, "shared": True, "force": path}
                 for B in BATCHES]
    for kind, (dim, data) in failing_trusses().items():
        jobs.append({"label": kind, "dim": dim, "data": data, "B": 13, "seed": 4, "shared": True})
    res = H.run_band_child(tmp, {"TB_SUBST_TILE": "1"}, jobs)
    return {(j["label"], j["B"]): r for j, r in zip(jobs, res)}


@pytest.mark.parametrize("label", LABELS)
def test_warp_per_load_case_kernel_every_band_width(label, tile1_runs):
    """TB_SUBST_TILE=1 forces k_band_subst<NB> on every system: against the reference and at a backward error of
    rounding level, batch-size independent, and within 1e-12 of the default route (which sums in another order) on the
    well-conditioned systems."""
    s = system(label)
    F, want = reference_cases(label)
    print(f"{label}: {tile1_runs[label, NB_CASES][1]}")
    for B in BATCHES:
        out, seen = tile1_runs[label, B]
        assert H.subst_kernels(seen) == [f"k_band_subst<{s.NB}>"] and H.band_kernels(seen) == [s.factor], (B, seen)
        s.check(out, F[:B], {k: v[:B] for k, v in want.items() if k != "weight"} | {"weight": want["weight"]}, f"{label} B={B}")
        assert_same(out, {k: v[:B] for k, v in tile1_runs[label, NB_CASES][0].items()}, f"{label} B={B}")
    dflt = default_runs(label)[NB_CASES][0]
    tol = 1e-10 if label == "bar-942" else 1e-12        # cond(K_ff): 6e6 on bar-942, at most 6e5 on the others
    for k in H.FIELDS:
        assert orc.normwise_err(tile1_runs[label, NB_CASES][0][k], dflt[k]) <= tol, k


# --------------------------------------------------------------------------- every row of the factor
@pytest.mark.parametrize("label", ["t2d-4x41", "t3d-21x7", "ladder"])
def test_unit_loads_give_the_inverse(label):
    """A unit load on each free DOF in turn, and one zero load case: the free part of u is the matching column of
    K_ff^-1 (1e-9 norm-wise per column, backward error of rounding level), which reaches every row of every block,
    padding rows included; the zero load case gives exactly zero u, ext and axial."""
    s = system(label)
    dofs = np.nonzero(s.mask)[0]
    F = np.zeros((len(dofs) + 1, s.N))
    F[np.arange(len(dofs)), dofs] = 1.0
    out, seen = H.cuda_kernels(lambda: s.solve(F))
    print(f"{label}: {seen}")
    assert H.subst_kernels(seen) == [s.subst], seen
    assert not out["info"].any()
    inv = np.linalg.inv(s.Kff)
    got = out["u"][:-1][:, dofs].T
    err = np.abs(got - inv).max(axis=0) / np.abs(inv).max(axis=0)
    assert err.max() <= 1e-9, f"column {int(err.argmax())}: {err.max():.2e}"
    be = s.backward_errors(F[:-1], out["u"][:-1])
    assert be.max() <= BE_TOL, f"column {int(be.argmax())}: backward error {be.max():.2e}"
    for k in ("u", "ext", "axial"):
        assert not out[k][-1].any(), k


# --------------------------------------------------------------------------- bit identity
@pytest.mark.parametrize("label", ["bar-6", "t2d-4x40", "t3d-10x14", "t3d-21x7", "ladder"])
def test_load_case_bits_do_not_depend_on_its_neighbours(label):
    """One load case alone, at every position of a tile of eight (k_band_subst8) or a CTA of four (k_band_subst), in
    the first tile and the second, with other load cases around it each time: the same bits everywhere."""
    s = system(label)
    x = s.loads(1, seed=7)
    solo, seen = H.cuda_kernels(lambda: s.solve(x))
    assert H.subst_kernels(seen) == [s.subst], seen
    for pos in range(16):
        F = s.loads(pos + 1 + (pos % 3), seed=100 + pos)
        F[pos] = x[0]
        out = s.solve(F)
        assert_same({k: v[pos:pos + 1] for k, v in out.items()}, solo, f"{label} position {pos} of {F.shape[0]}")


@pytest.mark.parametrize("label", ["t2d-4x40", "bar-942", "t3d-21x7", "bar-10", "ladder"])
def test_one_case_batch_equals_its_place_in_a_larger_batch(label):
    """loadcases(F[j:j+1]) is loadcases(F)[j], bit for bit: a batch of one takes the shared route too."""
    s = system(label)
    F, _ = reference_cases(label)
    whole = default_runs(label)[NB_CASES][0]
    for j in (0, 8, NB_CASES - 1):
        one, seen = H.cuda_kernels(lambda: s.solve(F[j:j + 1]))
        assert H.subst_kernels(seen) == [s.subst] and H.band_kernels(seen) == [s.factor], seen
        assert_same(one, {k: v[j:j + 1] for k, v in whole.items()}, f"{label} case {j}")


def test_tile_kernel_grid_stride_bar942():
    """More tiles than k_band_subst8's grid (SMs * floor(220 KB / (smem8 + 1 KB)) CTAs): CTAs loop over several tiles,
    the last one partial.  Slices across the first tile, the grid-stride boundary and the end, solved as small batches,
    give the same bits; samples against the reference."""
    s = system("bar-942")
    cap = n_sm() * ((220 * 1024) // (s.smem8 + 1024))
    B = 8 * cap + 8 * 3 + 5
    assert (B + 7) // 8 > cap and s.subst == f"k_band_subst8<{s.NB}>"
    F = s.loads(B, seed=21)
    out, seen = H.cuda_kernels(lambda: s.solve(F))
    print(f"bar-942 x{B} (grid cap {cap} tiles): {seen}")
    assert H.subst_kernels(seen) == [s.subst] and seen[s.subst] == 1, seen
    assert not out["info"].any()
    for lo, hi in ((0, 9), (8 * cap - 3, 8 * cap + 14), (B - 13, B)):
        assert_same(s.solve(F[lo:hi]), {k: v[lo:hi] for k, v in out.items()}, f"[{lo}:{hi}]")
    pick = np.array([0, 8 * cap - 1, 8 * cap, B - 1])
    s.check({k: v[pick] for k, v in out.items()}, F[pick], s.reference(F[pick]), "bar-942 grid-stride")


# --------------------------------------------------------------------------- entry points and chunking
@pytest.mark.parametrize("label", ["bar-942", "ladder"])
def test_host_entry_point_and_compact_outputs(label):
    """tb_solve_loadcases_host gives the device call's bits; the compact outputs (u_free, react) of a shared call are
    the dense ones, through both entry points."""
    s = system(label)
    torch = _torch()
    F, _ = reference_cases(label)
    dense = default_runs(label)[NB_CASES][0]
    host = s.plan.solve_host(NB_CASES, s.joints, F, aed=s.aed, shared_factor=True)
    assert_same(host, dense, f"{label} host")
    free_idx, _, sup_idx = s.plan.maps()
    dev = torch.device("cuda:0")
    td = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    f64 = dict(dtype=torch.float64, device=dev)
    out = {"u_free": torch.empty(NB_CASES, s.n, **f64), "react": torch.empty(NB_CASES, s.plan.s, **f64),
           "axial": torch.empty(NB_CASES, s.M, **f64), "info": torch.empty(NB_CASES, dtype=torch.int32, device=dev)}
    s.plan.solve_device(NB_CASES, td(s.joints), td(F), aed=td(s.aed), out=out, shared_factor=True)
    torch.cuda.synchronize()
    compact = {k: v.cpu().numpy() for k, v in out.items()}
    hcompact = s.plan.solve_host(NB_CASES, s.joints, F, aed=s.aed, want=("u_free", "react", "axial"), shared_factor=True)
    for got in (compact, hcompact):
        assert np.array_equal(got["u_free"], dense["u"][:, free_idx]) and np.array_equal(got["react"], dense["ext"][:, sup_idx])
        assert np.array_equal(got["axial"], dense["axial"]) and not got["info"].any()


def test_chunked_calls_give_the_device_bits(tmp_path):
    """The host entry point cut into three chunks (TB_HOST_CHUNKS=3: 3 and 4 load cases leave chunks of one), and the
    device entry point cut at a 0.25 GB workspace (TB_WORKSPACE_MAX_GB, bar-942: 251 load cases per chunk, the last
    chunk one load case, each chunk factorising its first load case again): the bits of one unchunked device call."""
    jobs, want = [], []
    for label in ("bar-942", "ladder"):
        s = system(label)
        F, _ = reference_cases(label)
        path = str(tmp_path / f"{label}.npy")
        np.save(path, F)
        for B in (3, 4, NB_CASES):
            jobs.append({"label": label, "dim": s.dim, "data": s.data, "B": B, "seed": 0, "shared": True, "host": True,
                         "force": path})
            want.append(s.solve(F[:B]))
    for (got, _), job, w in zip(H.run_band_child(tmp_path, {"TB_HOST_CHUNKS": "3"}, jobs), jobs, want):
        assert_same(got, w, f"{job['label']} host chunks B={job['B']}")

    s = system("bar-942")
    prog = s.plan.ts_program()["info"]
    d = s.dim
    per = s.M * (2 + d + d * (d + 1) // 2) + s.plan.info.nnz_lower + s.nb16 * (s.NB + 1) * 256 + s.nb16 * 256 + s.nb16 * 16
    ts = (prog["l_per_sys"] + prog["nS"] ** 2 * 64 + prog["nS"] * 8 + prog["n_pad"] + len(s.plan.ts_program()["epos"])) * 8 + 4 + 4096
    per_sys = ((per * 8 + 4 + 1024 + 255) & ~255) + ts           # plan_ws_bytes(p, 1): csrc/tb_api.cu, csrc/tb_large.cu
    chunk = (1 << 28) // per_sys
    B = 4 * chunk + 1
    F = s.loads(B, seed=31)
    path = str(tmp_path / "bar-942_ws.npy")
    np.save(path, F)
    (got, seen), = H.run_band_child(tmp_path, {"TB_WORKSPACE_MAX_GB": "0.25"}, [
        {"label": "bar-942", "dim": s.dim, "data": s.data, "B": B, "seed": 0, "shared": True, "force": path}])
    print(f"bar-942 x{B} in chunks of {chunk}: {seen}")
    assert seen.get("k_prep<3>") == 5 and seen.get(s.factor) == 5 and seen.get(s.subst) == 5, seen
    assert_same(got, s.solve(F), f"bar-942 x{B} workspace chunks")


# --------------------------------------------------------------------------- failures
@functools.lru_cache(maxsize=None)
def failing_trusses():
    """t3d-5x24 with every member of zero stiffness (the factorisation fails) and with a zero-length member."""
    dim, data = systems()["t3d-5x24"]
    no_e = json.loads(json.dumps(data))
    for m in no_e["member"]:
        m[1][1] = 0.0
    zero_len = json.loads(json.dumps(data))
    j0, j1 = zero_len["member"][0][0]
    zero_len["joint"][j1][0] = list(zero_len["joint"][j0][0])
    assert zero_len["joint"][j1][1] == "NO"
    return {"zero-stiffness": (dim, no_e), "zero-length": (dim, zero_len)}


@pytest.mark.parametrize("kind", ["zero-stiffness", "zero-length"])
def test_shared_factor_failures(kind, tile1_runs):
    """A failed factorisation (info > 0) or input (a zero-length member: the info of the independent call) reaches
    every one of 13 load cases with zero outputs, under both substitution kernels."""
    dim, data = failing_trusses()[kind]
    s = System(kind, dim, data, dense=False)
    F = BC.inputs(s.plan, BC.Entry(kind, dim, data, {}), 13, seed=4)[2]
    out, seen = H.cuda_kernels(lambda: s.solve(F))
    indep = H.solve_device_np(s.plan, 13, s.joints, s.aed, F)
    print(f"{kind}: info {int(out['info'][0])} (independent {sorted(set(indep['info'].tolist()))}), {seen}")
    for what, (res, tags), kernel in (("default", (out, seen), s.subst), ("TB_SUBST_TILE=1", tile1_runs[kind, 13], f"k_band_subst<{s.NB}>")):
        assert H.subst_kernels(tags) == [kernel], (what, tags)
        info = res["info"]
        assert len(set(info.tolist())) == 1 and info[0] != 0, (what, info)
        if kind == "zero-stiffness":
            assert info[0] > 0, (what, info)
        else:
            assert np.array_equal(info, indep["info"]), (what, info, indep["info"])
        for k in ("u", "ext", "axial", "weight"):
            assert not res[k].any(), (what, k)


# --------------------------------------------------------------------------- reverse mode
def test_shared_factor_adjoint_on_the_ladder():
    """The shared-factor adjoint through k_band_subst against the independent adjoint (1e-10) and oracle/adjoint.py."""
    s = system("ladder")
    B = 3
    F = s.loads(B, seed=5)
    grads = random_grads(np.random.default_rng(5), B, s.N, s.M)
    (_, shared), seen = H.cuda_kernels(lambda: device_adjoint(s.plan, s.joints, s.aed, F, grads, shared_factor=True))
    print(f"ladder adjoint: {seen}")
    assert H.subst_kernels(seen) == [s.subst] and s.subst.startswith("k_band_subst<"), seen
    _, indep = device_adjoint(s.plan, s.joints, s.aed, F, grads)
    assert not shared["info"].any() and not indep["info"].any()
    for k in GRAD_FIELDS:
        for b in range(B):
            assert orc.normwise_err(shared[k][b], indep[k][b]) <= 1e-10, (k, b)
    for b in (0, 2):
        assert_grads_close(shared, oracle_grads(s.dim, s.joints, s.support, s.conn, s.aed, F[b], grads, b), b, what="ladder")
