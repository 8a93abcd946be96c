"""Host-side mirror of the slice of ``tbmodels.Model`` that the k-space hot path touches.

``KModel`` carries exactly the state ``Model.hamilton`` / ``Model.eigenval`` read -- ``hop`` (half-set dict),
``pos``, ``size``, ``dim`` (reference src/tbmodels/_tb_model.py:186-218) -- and exposes the same two methods
with the same signatures, return types and error behaviour (:1076-1150), evaluated on the GPU.

It exists so that (a) the accelerated path can be used and tested on machines where the reference package
is not installed (the GPU box), and (b) a ``tbmodels.Model`` can be handed over with
``KModel.from_model(model)``.  Model construction / file formats / model algebra stay in the reference.
"""
from __future__ import annotations

import numpy as np

from ._evaluator import Evaluator
from ._pack import PackedModel, hop_dict, pack_arrays, pack_model


class KModel:
    """Duck-type of ``tbmodels.Model`` restricted to the k-space evaluation path."""

    def __init__(self, *, hop, pos, size=None, dim=None, device=None):
        pos = np.array(pos, dtype=float)
        self.size = int(size) if size is not None else pos.shape[0]
        self.dim = int(dim) if dim is not None else pos.shape[1]
        self.pos = pos.reshape(self.size, self.dim)
        self.hop = {tuple(int(x) for x in R): np.array(mat, dtype=complex) for R, mat in hop.items()}
        self.uc = None
        self.occ = None
        self._device = device
        self._cache = None  # (digest, Evaluator); never pickled

    # -- constructors ------------------------------------------------------------------------------
    @classmethod
    def from_packed(cls, packed: PackedModel, device=None) -> "KModel":
        return cls(hop=hop_dict(packed), pos=packed.pos, size=packed.size, dim=packed.dim, device=device)

    @classmethod
    def from_arrays(cls, R, hop, pos, device=None) -> "KModel":
        return cls.from_packed(pack_arrays(R, hop, pos), device=device)

    @classmethod
    def from_model(cls, model, device=None) -> "KModel":
        """Snapshot of a ``tbmodels.Model`` (or anything with hop / pos / size / dim)."""
        return cls.from_packed(pack_model(model), device=device)

    # -- pickling: device handles never enter the pickled state (reference tests/test_pickle.py) -------
    def __getstate__(self):
        state = dict(self.__dict__)
        state["_cache"] = None
        return state

    # -- evaluation --------------------------------------------------------------------------------
    def evaluator(self) -> Evaluator:
        """Device copy of the current hoppings; re-packed when ``hop`` / ``pos`` were mutated."""
        packed = pack_model(self)
        digest = packed.digest()
        if self._cache is None or self._cache[0] != digest:
            if self._cache is not None:
                self._cache[1].close()
            self._cache = (digest, Evaluator(packed, device=self._device))
        return self._cache[1]

    def hamilton(self, k, convention=2):
        """Same contract as ``tbmodels.Model.hamilton`` (reference :1076-1132)."""
        if convention not in [1, 2]:
            raise ValueError(
                "Invalid value '{}' for 'convention': must be either '1' or '2'".format(convention)
            )
        return self.evaluator().hamilton(k, convention=convention)

    def eigenval(self, k):
        """Same contract as ``tbmodels.Model.eigenval`` (reference :1134-1150)."""
        return self.evaluator().eigenval(k)

    def construct_kdotp(self, k, order: int):
        """Same contract as ``tbmodels.Model.construct_kdotp`` (reference :942-982); returns a :class:`KdotpModel`."""
        from ._kdotp import KdotpModel

        return KdotpModel(self.evaluator().construct_kdotp(k, order), device=self._device)

    def eigh(self, k):
        """Eigenvalues and eigenvectors of the convention-2 H(k) (extension, see :meth:`Evaluator.eigh`)."""
        return self.evaluator().eigh(k)

    def band_velocity(self, k, degen_tol=1e-8):
        """Eigenvalues and band velocities dE/dk of the convention-2 H(k) (extension, see :meth:`Evaluator.band_velocity`)."""
        return self.evaluator().band_velocity(k, degen_tol=degen_tol)

    def berry_curvature(self, k, convention=2, degen_tol=1e-8):
        """Eigenvalues and Berry curvature of every band (extension, see :meth:`Evaluator.berry_curvature`)."""
        return self.evaluator().berry_curvature(k, convention=convention, degen_tol=degen_tol)

    def supercell(self, size) -> "SupercellKModel":
        """``Model.supercell(size)`` (reference :1645-1724) evaluated without building the supercell's dense hopping
        matrices: see :meth:`Evaluator.from_supercell`."""
        return SupercellKModel(pack_model(self), size, device=self._device)


class SupercellKModel:
    """Supercell of a packed base model, device-packed (SURVEY.md section 8 f3).  Duck-type of the evaluated part of
    ``tbmodels.Model``: ``size``, ``dim``, ``pos`` plus ``hamilton`` / ``eigenval`` / ``eigh`` / ``band_velocity`` /
    ``berry_curvature``.  There is no ``hop`` dict --
    build the supercell with the reference's ``Model.supercell`` when the dense matrices themselves are needed."""

    def __init__(self, base: PackedModel, size, device=None):
        import itertools

        size_arr = np.array(size).astype(dtype=int, casting="safe")
        if size_arr.shape != (base.dim,):
            raise ValueError("The given 'size' has incorrect shape {}, should be {}.".format(size_arr.shape, (base.dim,)))
        if np.any(size_arr < 1):
            raise ValueError("supercell sizes must be >= 1")
        self.base = base
        self.supercell_size = tuple(int(x) for x in size_arr)
        self.dim = base.dim
        self.size = base.size * int(np.prod(size_arr))
        reduced = base.pos / size_arr  # reference :1670-1678
        self.pos = np.concatenate([reduced + np.array(off) / size_arr
                                   for off in itertools.product(*[range(n) for n in size_arr])])
        self._device = device
        self._ev = None

    def __getstate__(self):
        state = dict(self.__dict__)
        state["_ev"] = None
        return state

    def evaluator(self) -> Evaluator:
        if self._ev is None:
            self._ev = Evaluator.from_supercell(self.base, self.supercell_size, device=self._device)
        return self._ev

    def hamilton(self, k, convention=2):
        if convention not in [1, 2]:
            raise ValueError("Invalid value '{}' for 'convention': must be either '1' or '2'".format(convention))
        return self.evaluator().hamilton(k, convention=convention)

    def eigenval(self, k):
        return self.evaluator().eigenval(k)

    def eigh(self, k):
        return self.evaluator().eigh(k)

    def band_velocity(self, k, degen_tol=1e-8):
        return self.evaluator().band_velocity(k, degen_tol=degen_tol)

    def berry_curvature(self, k, convention=2, degen_tol=1e-8):
        return self.evaluator().berry_curvature(k, convention=convention, degen_tol=degen_tol)
