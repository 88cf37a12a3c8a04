"""Bulk I/O for solved datasets (SURVEY.md section 8 f-3): the packed SoA arrays a ragged batch is solved in
(``tb_ragged_in`` / ``tb_batch_out`` layout, what ``GenerateAugmentedDataset`` and ``pack_ragged`` produce) as ONE
binary container instead of one JSON file per truss, plus the views back into the reference's formats:

* ``PackedDataset.from_json_files``   N reference JSON files -> packed arrays through the native parser (no Truss objects);
* ``PackedDataset.solve``             the whole container as one ragged GPU batch, results attached to the arrays;
* ``PackedDataset.solve_modes``       natural frequencies and mode shapes of every truss in one ragged GPU batch;
* ``PackedDataset.save / load``       one ``.npz`` (optionally compressed) holding every array;
* ``PackedDataset.json(i)``           truss ``i`` as the reference's JSON dict (``Truss.Serialize``, truss.py:367-395 and
                                      ``detail/combine_with_JSON.md:71-163``: sparse ``displace / external / internal`` lists
                                      under the 1e-10 filter of truss.py:344-361), built straight from the arrays;
* ``PackedDataset.truss(i)``          a ``Truss`` object with the results attached (getters work, no re-solve);
* ``PackedDataset.dump_json(folder)`` the reference's one-file-per-truss layout (generate.py:361-362), for consumers
                                      that read it.
The reference writes and reads only per-truss JSON (``Truss.DumpIntoJSON / LoadFromJSON``).
"""
from __future__ import annotations

import json
import os

import numpy as np

from .type import SupportType
from .utils import CheckDim, ZERO_EPS

_ARRAYS = ("joint_off", "member_off", "xyz", "support", "conn", "aed", "force")
_RESULTS = ("u", "ext", "axial", "weight", "info")
_MODES = ("eigval", "modes", "n_free", "modes_info")   # solve_modes: [B, k], [k d sum nJ], [B], [B]
_SUPPORT_NAMES = {int(v): SupportType.GetFromType(v) for v in (SupportType.NO, SupportType.PIN, SupportType.ROLLER_X,
                                                               SupportType.ROLLER_Y, SupportType.ROLLER_Z)}


class PackedDataset:
    """B trusses packed back to back: truss ``i`` owns joints ``joint_off[i]:joint_off[i+1]`` and members
    ``member_off[i]:member_off[i+1]``; ``conn`` holds local joint ids; ``u / ext / force`` are ``dim`` per joint."""

    def __init__(self, dim, arrays: dict, names=None):
        self.dim = int(dim)
        self.a = {k: np.asarray(arrays[k]) for k in _ARRAYS}
        for k in _RESULTS + _MODES + ("src",):
            if k in arrays and arrays[k] is not None:
                self.a[k] = np.asarray(arrays[k])
        self.names = list(names) if names is not None else None
        jo, mo = self.a["joint_off"], self.a["member_off"]
        if jo.shape != mo.shape or jo[0] != 0 or mo[0] != 0:
            raise ValueError("joint_off / member_off must be [B+1] prefix sums starting at 0")
        if self.a["xyz"].size != jo[-1] * self.dim or self.a["conn"].size != 2 * mo[-1] or self.a["aed"].size != 3 * mo[-1]:
            raise ValueError("array sizes do not match the offsets")

    def __len__(self):
        return int(self.a["joint_off"].shape[0] - 1)

    @property
    def solved(self):
        return all(k in self.a for k in ("u", "ext", "axial"))

    @classmethod
    def from_trusses(cls, trusses, names=None):
        """Pack Truss objects (results included when every truss is solved)."""
        from .batch import pack_ragged
        trusses = list(trusses)
        dim, jo, mo, xyz, sup, conn, aed, force = pack_ragged(trusses)
        arrays = {"joint_off": jo, "member_off": mo, "xyz": xyz, "support": sup, "conn": conn, "aed": aed, "force": force}
        if all(t.isSolved for t in trusses):
            arrays["u"] = np.concatenate([t._dense_or_from_sparse("u") for t in trusses])
            arrays["ext"] = np.concatenate([t._dense_or_from_sparse("ext") for t in trusses])
            arrays["axial"] = np.concatenate([t._dense_or_from_sparse("axial") for t in trusses])
            arrays["weight"] = np.array([t.weight for t in trusses])
            arrays["info"] = np.zeros(len(trusses), np.int32)
        return cls(dim, arrays, names)

    @classmethod
    def from_json_texts(cls, texts, dim, isOutputFile=False, names=None, threads=0):
        """Pack JSON documents of the reference's format (``bytes``) without building Truss objects: the bulk form of
        ``Truss(dim).LoadFromJSON(path, isOutputFile)`` (truss.py:401-421), parsed by the native loader
        (csrc/tb_json.cu) on ``threads`` host threads (0: all cores).  Raises ValueError naming the first bad document."""
        from . import _lib
        from .utils import InvaildJointError, InvalidSupportTypeError
        arrays, err = _lib.json_load_packed(list(texts), CheckDim(dim), isOutputFile, threads)
        bad = np.nonzero(err)[0]
        if bad.size:
            i, code = int(bad[0]), int(err[bad[0]])
            who = names[i] if names is not None else f"document {i}"
            if code == -5:
                raise InvalidSupportTypeError(f"[GetFromString] No such support type in {who} !")
            if code == -4:
                raise InvaildJointError(f"{who}: a load, member or result entry refers to a joint / member that does not exist.")
            raise ValueError(f"{who}: not a truss JSON document ({_lib.strerror(code)})")
        if isOutputFile:
            arrays["info"] = np.zeros(len(err), np.int32)
            if np.isnan(arrays["weight"]).any():           # ("weight" is optional in the files: a * L * density summed, truss.py:166-168)
                xyz = arrays["xyz"].reshape(-1, dim)
                conn = arrays["conn"].reshape(-1, 2).astype(np.int64)
                owner = np.repeat(np.arange(len(err)), np.diff(arrays["member_off"]))      # truss of every member
                base = arrays["joint_off"][:-1][owner]
                length = np.sqrt(((xyz[base + conn[:, 1]] - xyz[base + conn[:, 0]]) ** 2).sum(axis=1))
                aed = arrays["aed"].reshape(-1, 3)
                w = np.bincount(owner, weights=aed[:, 0] * length * aed[:, 2], minlength=len(err))
                arrays["weight"] = np.where(np.isnan(arrays["weight"]), w, arrays["weight"])
        return cls(dim, arrays, names)

    @classmethod
    def from_json_files(cls, paths, dim, isOutputFile=False, threads=0):
        """``from_json_texts`` over files; truss ``i`` is named after file ``i`` (without the extension)."""
        paths = list(paths)
        texts = []
        for p in paths:
            with open(p, "rb") as f:
                texts.append(f.read())
        return cls.from_json_texts(texts, dim, isOutputFile, [os.path.splitext(os.path.basename(p))[0] for p in paths], threads)

    def solve(self, raise_on_error=False):
        """Solve every truss of the container in one ragged GPU batch (tb_solve_ragged_host; the bulk form of the
        generator's solve site generate.py:354-357) and attach ``u / ext / axial / weight / info`` -- no Truss objects.
        Returns the per-truss info codes (0 solved, -1 fails the counting rule, k > 0 singular at pivot k)."""
        from . import _lib
        from .truss import raise_for_info
        a = self.a
        out = _lib.solve_ragged_host(self.dim, a["joint_off"], a["member_off"], a["xyz"], a["support"], a["conn"], a["aed"], a["force"])
        for k in _RESULTS:
            self.a[k] = out[k]
        if raise_on_error:
            bad = np.nonzero(out["info"])[0]
            if bad.size:
                raise_for_info(int(out["info"][bad[0]]))
        return out["info"]

    def solve_modes(self, nMode, isConsistentMass=False, jointMasses=None):
        """The ``nMode`` lowest eigenpairs of every truss in one ragged GPU batch (tb_modes_ragged_host) -- labels for
        surrogates of generated trusses -- attached as ``eigval`` [B, nMode] (lambda = omega^2, ascending), ``modes``
        [nMode d sum nJ] (truss i's block [nMode][d nJ_i] starts at nMode d joint_off[i]), ``n_free`` [B] (entries past a
        truss's free-DOF count are 0) and ``modes_info`` [B] (status codes of tb_modes).  ``jointMasses``: None or
        [sum nJ] non-structural mass per joint.  Returns ``modes_info``."""
        from . import _lib
        a = self.a
        out = _lib.modes_ragged_host(self.dim, a["joint_off"], a["member_off"], a["xyz"], a["support"], a["conn"], a["aed"],
                                     int(nMode), consistent=isConsistentMass, joint_mass=jointMasses)
        for k in ("eigval", "modes", "n_free"):
            self.a[k] = out[k]
        self.a["modes_info"] = out["info"]
        return out["info"]

    # ------------------------------------------------------------------ binary container
    def save(self, path, compressed=False):
        payload = dict(self.a)
        payload["dim"] = np.int32(self.dim)
        if self.names is not None:
            payload["names"] = np.array(self.names)
        (np.savez_compressed if compressed else np.savez)(path, **payload)
        return path

    @classmethod
    def load(cls, path):
        with np.load(path, allow_pickle=False) as z:
            arrays = {k: z[k] for k in z.files if k not in ("dim", "names")}
            names = [str(s) for s in z["names"]] if "names" in z.files else None
            return cls(int(z["dim"]), arrays, names)

    # ------------------------------------------------------------------ views in the reference's formats
    def _range(self, i):
        jo, mo = self.a["joint_off"], self.a["member_off"]
        return int(jo[i]), int(jo[i + 1]), int(mo[i]), int(mo[i + 1])

    def json(self, i):
        """Truss ``i`` as the dict ``Truss.Serialize()`` returns (truss.py:384-395)."""
        d = self.dim
        j0, j1, m0, m1 = self._range(i)
        xyz = self.a["xyz"][d * j0:d * j1].reshape(-1, d)
        force = self.a["force"][d * j0:d * j1].reshape(-1, d)
        conn = self.a["conn"][2 * m0:2 * m1].reshape(-1, 2)
        aed = self.a["aed"][3 * m0:3 * m1].reshape(-1, 3)
        data = {"joint": [[row.tolist(), _SUPPORT_NAMES[int(s)]] for row, s in zip(xyz, self.a["support"][j0:j1])],
                "force": [[int(j), force[j].tolist()] for j in np.nonzero(force.any(axis=1))[0]],
                "member": [[[int(c[0]), int(c[1])], row.tolist()] for c, row in zip(conn, aed)]}
        if self.solved and ("info" not in self.a or self.a["info"][i] == 0):
            u = self.a["u"][d * j0:d * j1].reshape(-1, d)
            ext = self.a["ext"][d * j0:d * j1].reshape(-1, d)
            ax = self.a["axial"][m0:m1]
            keep = lambda rows: np.nonzero(~(np.abs(rows) < ZERO_EPS).all(axis=1))[0]  # noqa: E731  (truss.py:344-351)
            data["displace"] = [[int(j), u[j].tolist()] for j in keep(u)]
            data["external"] = [[int(j), ext[j].tolist()] for j in keep(ext)]
            data["internal"] = [[int(m), float(ax[m])] for m in np.nonzero(~(np.abs(ax) < ZERO_EPS))[0]]
            data["weight"] = float(self.a["weight"][i])
        return data

    def truss(self, i):
        """Truss ``i`` as a Truss object; solved results are attached without solving again."""
        from .truss import Truss
        d = self.dim
        j0, j1, m0, m1 = self._range(i)
        t = Truss(d).LoadFromJSON(data={k: v for k, v in self.json(i).items() if k in ("joint", "force", "member")})
        if self.solved and ("info" not in self.a or self.a["info"][i] == 0):
            t._set_dense_results(self.a["u"][d * j0:d * j1], self.a["ext"][d * j0:d * j1], self.a["axial"][m0:m1])
        if "eigval" in self.a and self.a["modes_info"][i] == 0:
            k, q = self.a["eigval"].shape[1], int(self.a["n_free"][i])
            block = self.a["modes"][k * d * j0:k * d * j1].reshape(k, d * (j1 - j0))
            t._modes = {"eigval": self.a["eigval"][i, :min(k, q)].copy(), "modes": block[:min(k, q)].copy()}
        return t

    def dump_json(self, folder, indices=None):
        """One JSON file per truss, the layout GenerateRandomCubeTrusses(saveFolder=...) writes (generate.py:361-362)."""
        os.makedirs(folder, exist_ok=True)
        paths = []
        for i in (range(len(self)) if indices is None else indices):
            name = self.names[i] if self.names is not None else f"truss_{i}"
            paths.append(os.path.join(folder, name + ".json"))
            with open(paths[-1], "w", encoding="utf-8") as f:
                json.dump(self.json(i), f)
        return paths
