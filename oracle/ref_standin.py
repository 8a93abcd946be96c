"""TEST INFRASTRUCTURE ONLY -- stand-in for the reference ``tbmodels`` package where its sources are absent.

``tests/test_gpu_reference_class.py`` switches the GPU methods onto ``tbmodels.Model`` with ``tbmodels_b200.install()``.
When the unmodified reference cannot be imported (``oracle/ref_shim.py``), it installs them on this ``Model`` instead.
The class keeps the data the installed methods read exactly as the reference lays it out: the half-set ``hop`` dict
with half of the R = 0 block, csr matrices for ``sparse=True``, ``pos``, ``size`` and ``dim``.  Its construction rules
are the ones ``oracle/workloads.py`` and ``tbmodels_b200/io.py`` restate (``add_hop``, ``on_site``, ``contains_cc=False``
input, ``supercell``), and its numpy methods are the oracle's (``oracle/tb_oracle.py``).  tests/test_oracle_golden.py
pins both against outputs of the unmodified reference stored under ``tests/golden``.

The product package never imports this module.
"""
from __future__ import annotations

import types

import numpy as np
import scipy.sparse as sp

from oracle import tb_oracle as orc
from oracle import workloads as wl
from tbmodels_b200._pack import hop_dict, pack_model
from tbmodels_b200.io import _normalise_hop


class Model:
    """The part of ``tbmodels.Model`` (reference src/tbmodels/_tb_model.py) that the GPU tests exercise."""

    def __init__(self, *, on_site=None, hop=None, pos=None, occ=None, size=None, dim=None, sparse=False, contains_cc=True):
        pos = np.array(pos, dtype=float)
        self.size = int(size) if size is not None else pos.shape[0]
        self.dim = int(dim) if dim is not None else pos.shape[1]
        self.occ = occ
        self.sparse = bool(sparse)
        self._builder = wl.HopBuilder(self.size, self.dim, pos)
        if hop:
            if contains_cc:
                raise NotImplementedError("the stand-in takes hoppings only with contains_cc=False")
            hop, self._builder.pos = _normalise_hop({tuple(R): np.array(m, dtype=complex) for R, m in hop.items()},
                                                    self._builder.pos, self.size)
            self._builder.hop.update(hop)
        if on_site is not None:
            self._builder.add_on_site(on_site)

    @classmethod
    def _from_packed(cls, packed, sparse):
        model = cls(pos=packed.pos, size=packed.size, dim=packed.dim, sparse=sparse)
        model._builder.hop.update(hop_dict(packed))
        return model

    @property
    def pos(self):
        return self._builder.pos

    @property
    def hop(self):
        return {R: sp.csr_matrix(m) if self.sparse else m for R, m in self._builder.hop.items()}

    def add_hop(self, overlap, orbital_1, orbital_2, R):
        self._builder.add_hop(overlap, orbital_1, orbital_2, R)

    def hamilton(self, k, convention=2):
        p = pack_model(self)
        return orc.hamilton(p.R, p.hop, p.pos, k, convention)

    def eigenval(self, k):
        p = pack_model(self)
        return orc.eigenval(p.R, p.hop, p.pos, k)

    def construct_kdotp(self, k, order):
        p = pack_model(self)
        return KdotpModel(orc.construct_kdotp(p.R, p.hop, p.pos, k, order))

    def supercell(self, size):
        return Model._from_packed(wl.supercell(pack_model(self), size), self.sparse)

    def __add__(self, other):
        if (self.size, self.dim) != (other.size, other.dim) or not np.array_equal(self.pos, other.pos):
            raise ValueError("models must have the same size, dimension and positions")
        model = Model(pos=self.pos, size=self.size, dim=self.dim, sparse=self.sparse)
        for R in list(self._builder.hop) + [R for R in other._builder.hop if R not in self._builder.hop]:
            zero = np.zeros((self.size, self.size), dtype=complex)
            model._builder.hop[R] = self._builder.hop.get(R, zero) + other._builder.hop.get(R, zero)
        return model

    def __mul__(self, x):
        model = Model(pos=self.pos, size=self.size, dim=self.dim, sparse=self.sparse)
        model._builder.hop.update({R: x * m for R, m in self._builder.hop.items()})
        return model

    __rmul__ = __mul__


class KdotpModel:
    """``tbmodels.kdotp.KdotpModel`` (reference src/tbmodels/kdotp.py:19-100) with the oracle's numpy methods."""

    def __init__(self, taylor_coefficients):
        for mat in taylor_coefficients.values():
            if not np.allclose(mat, np.array(mat).T.conj()):
                raise ValueError(f"The provided Taylor coefficient {mat} is not hermitian")
        self.taylor_coefficients = {tuple(key): np.array(mat, dtype=complex) for key, mat in taylor_coefficients.items()}

    def hamilton(self, k):
        return orc.kdotp_hamilton(self.taylor_coefficients, k)

    def eigenval(self, k):
        return orc.kdotp_eigenval(self.taylor_coefficients, k)


kdotp = types.SimpleNamespace(KdotpModel=KdotpModel)  # the reference's ``tbmodels.kdotp`` module path
