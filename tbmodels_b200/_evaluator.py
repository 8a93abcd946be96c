"""Device evaluator: the object that owns a ``tbk_model`` handle and mirrors the reference call contract.

``Evaluator.hamilton`` / ``Evaluator.eigenval`` reproduce the argument handling and return types of
``Model.hamilton`` / ``Model.eigenval`` (reference src/tbmodels/_tb_model.py:1076-1150):

* ``convention not in [1, 2]`` -> ``ValueError`` with the reference's message, before any device work (:1097-1102);
* ``np.array(k, ndmin=1)``; a 1-D (or scalar) k is a single point and the leading axis is squeezed from the
  result (:1103-1108, :1130-1132);
* ``eigenval`` of a k-list returns a Python ``list`` of ``[N]`` arrays, of a single point one ``[N]`` array
  (:1148-1150).  The list elements are views of one ``[n_k, N]`` buffer (``eigenval_array`` returns it whole).

Everything numerical happens in libtbk.so; there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import weakref

import numpy as np

from . import _capi
from ._pack import PackedModel


def _check_convention(convention) -> int:
    if convention not in [1, 2]:
        raise ValueError(
            "Invalid value '{}' for 'convention': must be either '1' or '2'".format(convention)
        )
    return int(convention)


def _normalise_k(k, dim: int):
    """Reference semantics of ``k_array = np.array(k, ndmin=1)`` + single-point reshape (:1103-1108)."""
    k_array = np.asarray(k)  # same values as np.array(k, ndmin=1) at :1103, without copying a ready float64 array
    if k_array.ndim == 0:
        k_array = k_array.reshape((1,))
    if k_array.ndim == 1:
        single_point = True
        k_array = k_array.reshape((1, -1))
    else:
        single_point = False
    if k_array.ndim != 2:
        raise ValueError(f"k must be a k-point or a list of k-points, got an array of shape {k_array.shape}")
    if k_array.shape[1] != dim:
        # the reference fails inside np.dot(k_array, R) with a ValueError as well
        raise ValueError(
            f"shapes {k_array.shape} and ({dim},) not aligned: k-points must have {dim} component(s)"
        )
    if k_array.dtype.kind not in "fiub":
        raise TypeError(f"k-points must be real numbers, got dtype {k_array.dtype}")
    return np.ascontiguousarray(k_array, dtype=np.float64), single_point


def _check_degen_tol(degen_tol) -> float:
    tol = float(degen_tol)
    if not tol >= 0.0:
        raise ValueError(f"degen_tol must be a number >= 0, got {degen_tol!r}")
    return tol


def kdotp_powers(dim: int, order: int) -> np.ndarray:
    """Power tuples of a k.p expansion up to ``order`` in the reference's order (:963-966)."""
    import itertools

    keys = [p for p in itertools.product(range(order + 1), repeat=dim) if sum(p) <= order]
    return np.array(keys, dtype=np.int32).reshape(len(keys), dim)


def pinned_empty(shape, dtype=np.float64) -> np.ndarray:
    """Uninitialised page-locked numpy array (fast path of the host entry points); freed with the array."""
    lib = _capi.load()
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) if np.ndim(shape) else int(shape)
    nbytes = max(n * dtype.itemsize, 1)
    ptr = C.c_void_p()
    _capi.check(lib.tbk_host_alloc(C.byref(ptr), nbytes))
    buf = (C.c_char * nbytes).from_address(ptr.value)
    arr = np.frombuffer(buf, dtype=dtype, count=n).reshape(shape)
    weakref.finalize(buf, lib.tbk_host_free, ptr.value)
    return arr


class Evaluator:
    """GPU-resident copy of one packed model plus the launch plumbing.

    The handle owns ONE set of device scratch.  The ``*_device`` methods enqueue on torch's current stream and return
    without synchronising; libtbk orders every call behind the previous one on the device (an event recorded on the
    stream of each call, waited on by the next), so mixing ``*_device`` calls on different torch streams with the
    host-buffer methods (which run on private streams) is safe -- they serialise, they do not race.  Deferred errors of
    the asynchronous calls (QL non-convergence) surface at :meth:`check`."""

    def __init__(self, packed: PackedModel, device=None):
        self._lib = _capi.load()
        self.packed = packed
        self.size = packed.size
        self.dim = packed.dim
        if device is None:
            device = _default_device()
        self.device = int(device)
        handle = C.c_void_p()
        _capi.check(
            self._lib.tbk_model_create(
                packed.dim,
                packed.size,
                packed.n_R,
                packed.R.ctypes.data_as(C.c_void_p),
                packed.hop.ctypes.data_as(C.c_void_p),
                packed.pos.ctypes.data_as(C.c_void_p),
                self.device,
                C.byref(handle),
            )
        )
        self._handle = handle
        self._finalizer = weakref.finalize(self, self._lib.tbk_model_destroy, handle)

    @classmethod
    def from_kdotp(cls, powers, coeff, device=None) -> "Evaluator":
        """Evaluator of a k.p model ``H(k) = sum_q prod_d k_d^{p_qd} C_q`` (reference src/tbmodels/kdotp.py:51-100).

        ``powers`` int [n_terms, dim], ``coeff`` complex128 [n_terms, N, N] (Hermitian matrices).  ``hamilton`` must be
        called with the default ``convention=2`` (a k.p model has no orbital positions).
        """
        powers = np.ascontiguousarray(powers, dtype=np.int32)
        coeff = np.ascontiguousarray(coeff, dtype=np.complex128)
        if powers.ndim != 2 or coeff.ndim != 3 or coeff.shape[0] != powers.shape[0] or coeff.shape[1] != coeff.shape[2]:
            raise ValueError(f"inconsistent k.p arrays: powers {powers.shape}, coeff {coeff.shape}")
        self = cls.__new__(cls)
        self._lib = _capi.load()
        self.packed = None
        self.size = coeff.shape[1]
        self.dim = powers.shape[1]
        self.device = int(_default_device() if device is None else device)
        handle = C.c_void_p()
        _capi.check(
            self._lib.tbk_kdotp_create(
                self.dim,
                self.size,
                powers.shape[0],
                powers.ctypes.data_as(C.c_void_p),
                coeff.ctypes.data_as(C.c_void_p),
                self.device,
                C.byref(handle),
            )
        )
        self._handle = handle
        self._finalizer = weakref.finalize(self, self._lib.tbk_model_destroy, handle)
        return self

    @classmethod
    def from_supercell(cls, packed: PackedModel, size, device=None) -> "Evaluator":
        """Evaluator of ``Model.supercell(size)`` (reference src/tbmodels/_tb_model.py:1645-1724) built ON THE DEVICE from the
        base model's packed arrays (SURVEY.md section 8 f3): the dense ``[n_R', N', N']`` hopping tensor of the supercell is
        never materialised, and the H(k) GEMM skips the all-zero blocks of its weights."""
        size_arr = np.ascontiguousarray(np.array(size).astype(np.int32, casting="same_kind"))
        if size_arr.shape != (packed.dim,):
            raise ValueError(
                "The given 'size' has incorrect shape {}, should be {}.".format(size_arr.shape, (packed.dim,))
            )
        self = cls.__new__(cls)
        self._lib = _capi.load()
        self.packed = None
        self.dim = packed.dim
        self.size = packed.size * int(np.prod(size_arr))
        self.device = int(_default_device() if device is None else device)
        handle = C.c_void_p()
        _capi.check(
            self._lib.tbk_supercell_create(
                packed.dim, packed.size, packed.n_R, packed.R.ctypes.data_as(C.c_void_p),
                packed.hop.ctypes.data_as(C.c_void_p), packed.pos.ctypes.data_as(C.c_void_p),
                size_arr.ctypes.data_as(C.c_void_p), self.device, C.byref(handle),
            )
        )
        self._handle = handle
        self._finalizer = weakref.finalize(self, self._lib.tbk_model_destroy, handle)
        return self

    @property
    def lattice_vectors(self) -> np.ndarray:
        """The stored (half-set) lattice vectors of the handle, int32 ``[n_R, dim]`` in summation order."""
        n_R = C.c_int()
        _capi.check(self._lib.tbk_model_info(self._handle, None, None, C.byref(n_R), None))
        out = np.zeros((max(n_R.value, 1), self.dim), dtype=np.int32)
        _capi.check(self._lib.tbk_model_vectors(self._handle, out.ctypes.data_as(C.c_void_p)))
        return out[: n_R.value]

    # ------------------------------------------------------------------ info
    @property
    def path(self) -> str:
        p = C.c_int()
        _capi.check(self._lib.tbk_model_info(self._handle, None, None, None, C.byref(p)))
        return {0: "fused-small", 1: "gemm+tridiag-ql", 2: "fused-product"}[p.value]

    @property
    def launch_count(self) -> int:
        return int(self._lib.tbk_launch_count(self._handle))

    @property
    def workspace_bytes(self) -> int:
        return int(self._lib.tbk_workspace_bytes(self._handle))

    PROFILE_CLASSES = ("hk_gemm", "hk_small", "expand", "tridiag", "ql", "hk_phase", "mesh_lines", "eigh", "peer_push", "rescale")

    def profile(self, enable: bool = True) -> None:
        """Bracket every kernel launch with CUDA events on its stream (read back with :meth:`profile_read`)."""
        _capi.check(self._lib.tbk_profile(self._handle, 1 if enable else 0))

    def profile_read(self) -> dict:
        """``{class: (total_ms, launches)}`` accumulated since the last read (synchronises the device)."""
        ms = (C.c_double * len(self.PROFILE_CLASSES))()
        cnt = (C.c_int64 * len(self.PROFILE_CLASSES))()
        _capi.check(self._lib.tbk_profile_read(self._handle, ms, cnt))
        return {name: (float(ms[i]), int(cnt[i])) for i, name in enumerate(self.PROFILE_CLASSES)}

    # ------------------------------------------------------------------ regular k-meshes (no explicit k array)
    def _mesh_args(self, dims, shift):
        dims = [int(x) for x in np.atleast_1d(dims)]
        if len(dims) != self.dim or any(x < 1 for x in dims):
            raise ValueError(f"dims must hold {self.dim} positive mesh sizes")
        c_dims = (C.c_int64 * self.dim)(*dims)
        c_shift = None
        if shift is not None:
            shift = [float(x) for x in np.atleast_1d(shift)]
            if len(shift) != self.dim:
                raise ValueError(f"shift must hold {self.dim} values")
            c_shift = (C.c_double * self.dim)(*shift)
        n_lines_total = int(np.prod(dims[:-1])) if self.dim > 1 else 1
        return dims, c_dims, c_shift, n_lines_total

    def mesh_factorised(self, dims) -> bool:
        """True if :meth:`eigenval_mesh` will factorise the Fourier sum over the last mesh dimension for this model."""
        _, c_dims, _, _ = self._mesh_args(dims, None)
        return bool(self._lib.tbk_mesh_factorised(self._handle, c_dims))

    def eigenval_mesh_device(self, dims, shift=None, first_line=0, n_lines=None, out=None):
        """Eigenvalues on the regular mesh ``k_d = (i_d + shift_d) / dims[d]`` (``numpy.meshgrid(..., indexing="ij")``
        order), without an explicit k array: ``[n_lines * dims[-1], N]`` float64 CUDA tensor, asynchronous.

        ``first_line`` / ``n_lines`` select a contiguous range of lines (runs along the last dimension) for sharding.
        Same values as ``eigenval_device`` on the explicit mesh points, within the parity bounds."""
        import torch

        dims, c_dims, c_shift, total = self._mesh_args(dims, shift)
        if n_lines is None:
            n_lines = total - first_line
        n_k = int(n_lines) * dims[-1]
        if out is None:
            out = torch.empty((n_k, self.size), dtype=torch.float64, device=f"cuda:{self.device}")
        elif tuple(out.shape) != (n_k, self.size) or out.dtype != torch.float64 or not out.is_contiguous():
            raise ValueError("out must be a contiguous float64 tensor [n_lines * dims[-1], N]")
        _capi.check(
            self._lib.tbk_eigenval_mesh(
                self._handle, c_dims, c_shift, int(first_line), int(n_lines), C.c_void_p(out.data_ptr()), self._stream()
            )
        )
        return out

    def eigenval_mesh(self, dims, shift=None, first_line=0, n_lines=None, out=None) -> np.ndarray:
        """Eigenvalues on the regular mesh as a HOST array ``[n_lines * dims[-1], N]`` (default: the whole mesh) through
        ``tbk_eigenval_mesh_host``: groups of lines are evaluated into two device buffers whose D2H copies overlap the
        next group's kernels -- there is no k array to upload.  ``out`` may be a pinned buffer (:func:`pinned_empty`)."""
        dims, c_dims, c_shift, total = self._mesh_args(dims, shift)
        if n_lines is None:
            n_lines = total - first_line
        shape = (int(n_lines) * dims[-1], self.size)
        if out is None:
            out = np.empty(shape, dtype=np.float64)
        elif out.shape != shape or out.dtype != np.float64 or not out.flags.c_contiguous:
            raise ValueError("out must be a C-contiguous float64 array of shape %r" % (shape,))
        _capi.check(
            self._lib.tbk_eigenval_mesh_host(
                self._handle, c_dims, c_shift, int(first_line), int(n_lines), out.ctypes.data_as(C.c_void_p)
            )
        )
        return out

    def close(self) -> None:
        self._finalizer()

    def check(self) -> None:
        """Synchronise and raise if a device-pointer call hit a deferred error (QL non-convergence)."""
        _capi.check(self._lib.tbk_model_check(self._handle))

    # ------------------------------------------------------------------ host buffers (reference contract)
    def hamilton(self, k, convention=2, out=None):
        _check_convention(convention)
        k_array, single_point = _normalise_k(k, self.dim)
        n_k = k_array.shape[0]
        shape = (n_k, self.size, self.size)
        if out is None:
            out = np.empty(shape, dtype=np.complex128)
        elif out.shape != shape or out.dtype != np.complex128 or not out.flags.c_contiguous:
            raise ValueError("out must be a C-contiguous complex128 array of shape %r" % (shape,))
        _capi.check(
            self._lib.tbk_hamilton_host(
                self._handle,
                k_array.ctypes.data_as(C.c_void_p),
                n_k,
                int(convention),
                out.ctypes.data_as(C.c_void_p),
            )
        )
        if single_point:
            return out[0]
        return out

    def eigenval_array(self, k, out=None) -> np.ndarray:
        """Eigenvalues of a k-list as one ``[n_k, N]`` array (no per-k Python objects)."""
        k_array, _ = _normalise_k(k, self.dim)
        n_k = k_array.shape[0]
        shape = (n_k, self.size)
        if out is None:
            out = np.empty(shape, dtype=np.float64)
        elif out.shape != shape or out.dtype != np.float64 or not out.flags.c_contiguous:
            raise ValueError("out must be a C-contiguous float64 array of shape %r" % (shape,))
        _capi.check(
            self._lib.tbk_eigenval_host(
                self._handle, k_array.ctypes.data_as(C.c_void_p), n_k, out.ctypes.data_as(C.c_void_p)
            )
        )
        return out

    def eigenval(self, k):
        k_array, single_point = _normalise_k(k, self.dim)
        res = self.eigenval_array(k_array)
        if single_point:
            return res[0]
        return list(res)

    # ------------------------------------------------------------------ eigenvectors (SURVEY section 8 f4)
    def eigh(self, k):
        """Eigenvalues and eigenvectors of the convention-2 ``H(k)``: ``(w, v)`` like ``scipy.linalg.eigh`` applied to
        every ``Model.hamilton(k)[i]`` -- ``w`` ascending ``[n_k, N]``, ``v`` complex128 ``[n_k, N, N]`` with ``v[i][:, j]``
        the unit-norm eigenvector of ``w[i][j]`` (phase arbitrary).  A single k-point gives ``([N], [N, N])``."""
        k_array, single_point = _normalise_k(k, self.dim)
        n_k = k_array.shape[0]
        w = np.empty((n_k, self.size), dtype=np.float64)
        v = np.empty((n_k, self.size, self.size), dtype=np.complex128)
        _capi.check(
            self._lib.tbk_eigh_host(
                self._handle, k_array.ctypes.data_as(C.c_void_p), n_k, w.ctypes.data_as(C.c_void_p),
                v.ctypes.data_as(C.c_void_p),
            )
        )
        if single_point:
            return w[0], v[0]
        return w, v

    def eigh_device(self, k_dev, out_w=None, out_v=None):
        """Device-buffer form of :meth:`eigh`: float64 ``[n_k, dim]`` CUDA tensor -> ``(w [n_k, N], v [n_k, N, N])`` tensors,
        asynchronous on torch's current stream."""
        import torch

        k_dev = self._check_k_dev(k_dev)
        n_k = k_dev.shape[0]
        if out_w is None:
            out_w = torch.empty((n_k, self.size), dtype=torch.float64, device=k_dev.device)
        if out_v is None:
            out_v = torch.empty((n_k, self.size, self.size), dtype=torch.complex128, device=k_dev.device)
        if (tuple(out_w.shape) != (n_k, self.size) or out_w.dtype != torch.float64 or not out_w.is_contiguous()
                or tuple(out_v.shape) != (n_k, self.size, self.size) or out_v.dtype != torch.complex128
                or not out_v.is_contiguous()):
            raise ValueError("out_w / out_v must be contiguous float64 [n_k, N] / complex128 [n_k, N, N] tensors")
        _capi.check(
            self._lib.tbk_eigh(
                self._handle, C.c_void_p(k_dev.data_ptr()), n_k, C.c_void_p(out_w.data_ptr()),
                C.c_void_p(out_v.data_ptr()), self._stream(),
            )
        )
        return out_w, out_v

    # ------------------------------------------------------------------ band velocities dE/dk
    def band_velocity(self, k, degen_tol=1e-8):
        """Eigenvalues and band velocities of the convention-2 ``H(k)``: ``(w [n_k, N], v [n_k, N, dim])`` with
        ``w`` ascending (bit for bit what :meth:`eigh` returns) and ``v[i, n, d] = dE_n/dk_d`` at ``k[i]``.  A single
        k-point gives ``([N], [N, dim])``.

        ``k`` is in reduced coordinates, so ``v`` is in energy units per unit of reduced k; Cartesian velocities (per unit
        of Cartesian k, ``uc`` the lattice vectors as rows) are ``v @ uc / (2 pi)``.  Eigenvalues do not depend on the
        convention, so neither do their derivatives.

        * A band separated from its neighbours gets the Hellmann-Feynman value ``Re(v_n^H dH/dk_d v_n)``.
        * A degenerate cluster -- a maximal run of ascending eigenvalues whose consecutive gaps are
          ``<= degen_tol * rho``, ``rho = max_n |w_n|`` -- is treated as one level: per direction d separately, its
          members get the ascending eigenvalues of the block ``V_c^H dH/dk_d V_c`` (degenerate perturbation theory; the
          only choice independent of the basis eigh returns inside the subspace).  Inside a cluster the value at index n
          in direction 0 and the one at index n in direction 1 therefore need not belong to the same state.
        * ``degen_tol`` (>= 0, default 1e-8): an eigenvector with gap g is accurate to about ``eps rho / g``, so a pair
          left unmerged has a velocity error of at most about ``eps / degen_tol * ||dH/dk_d||`` (2e-8 of it at 1e-8),
          while a merged pair costs nothing: the block eigenvalues are exact for it.

        ``dH/dk_d`` is the order-1 term of :meth:`construct_kdotp`.  Not defined for k.p models (:class:`TbkError`)."""
        degen_tol = _check_degen_tol(degen_tol)
        k_array, single_point = _normalise_k(k, self.dim)
        n_k = k_array.shape[0]
        w = np.empty((n_k, self.size), dtype=np.float64)
        v = np.empty((n_k, self.size, self.dim), dtype=np.float64)
        _capi.check(
            self._lib.tbk_band_velocity_host(
                self._handle, k_array.ctypes.data_as(C.c_void_p), n_k, degen_tol, w.ctypes.data_as(C.c_void_p),
                v.ctypes.data_as(C.c_void_p),
            )
        )
        if single_point:
            return w[0], v[0]
        return w, v

    def band_velocity_device(self, k_dev, degen_tol=1e-8, out_w=None, out_v=None):
        """Device-buffer form of :meth:`band_velocity`: float64 ``[n_k, dim]`` CUDA tensor -> ``(w [n_k, N],
        v [n_k, N, dim])`` float64 tensors, asynchronous on torch's current stream."""
        import torch

        degen_tol = _check_degen_tol(degen_tol)
        k_dev = self._check_k_dev(k_dev)
        n_k = k_dev.shape[0]
        if out_w is None:
            out_w = torch.empty((n_k, self.size), dtype=torch.float64, device=k_dev.device)
        if out_v is None:
            out_v = torch.empty((n_k, self.size, self.dim), dtype=torch.float64, device=k_dev.device)
        if (tuple(out_w.shape) != (n_k, self.size) or out_w.dtype != torch.float64 or not out_w.is_contiguous()
                or tuple(out_v.shape) != (n_k, self.size, self.dim) or out_v.dtype != torch.float64
                or not out_v.is_contiguous()):
            raise ValueError("out_w / out_v must be contiguous float64 [n_k, N] / [n_k, N, dim] tensors")
        _capi.check(
            self._lib.tbk_band_velocity(
                self._handle, C.c_void_p(k_dev.data_ptr()), n_k, degen_tol, C.c_void_p(out_w.data_ptr()),
                C.c_void_p(out_v.data_ptr()), self._stream(),
            )
        )
        return out_w, out_v

    # ------------------------------------------------------------------ Berry curvature
    def berry_curvature(self, k, convention=2, degen_tol=1e-8):
        """Eigenvalues and Berry curvature of every band: ``(w [n_k, N], curv [n_k, N, P])``, ``P = dim (dim - 1) / 2``,
        with ``w`` ascending (bit for bit what :meth:`eigh` returns) and ``curv[i, n, p]`` the curvature
        ``Omega_n^{ab}`` at ``k[i]`` for the p-th pair ``a < b`` in the order (0,1), (0,2), ..., (0,dim-1), (1,2), ...
        (for dim = 3: ``Omega^01, Omega^02, Omega^12``).  A single k-point gives ``([N], [N, P])``.

        With ``V`` the eigenvectors, ``E = w`` and ``M_a = V^H X_a V``, ``X_a`` the k_a-derivative of H(k):

        * a band separated from its neighbours: ``Omega_n^{ab} = -2 Im sum_{l != n} M_a[n, l] M_b[l, n] /
          ((E_n - E_l)(E_n - E_l))``, the curl of the Berry connection ``A = i <u|grad u>``;
        * a degenerate cluster (as for :meth:`band_velocity`: a maximal run of ascending eigenvalues whose gaps are
          ``<= degen_tol * rho``, ``rho = max_n |w_n|``): per pair separately, its members get the ascending eigenvalues
          of the Hermitian non-Abelian curvature ``F_nm = i sum_{l not in c} (M_a[n, l] M_b[l, m] - M_b[n, l] M_a[l, m])
          / ((E_n - E_l)(E_m - E_l))``, whose trace is the sum of their Abelian curvatures and whose eigenvalues do not
          depend on the basis chosen inside the cluster;
        * ``convention`` (1 or 2, default 2 like :meth:`hamilton`): the local curvature depends on it, Chern numbers do
          not.  2: ``X_a = dH/dk_a`` (the order-1 term of :meth:`construct_kdotp`).  1: ``X_a = dH/dk_a + 2 pi i [H, T_a]``,
          ``T_a = diag(pos[:, a])``.

        ``k`` is in reduced coordinates, so ``curv`` is in units of (reduced k)^-2: ``sum_mesh curv[:, n, p] / n_k / (2
        pi)`` tends to the Chern number of band n, and the Cartesian tensor is ``uc.T @ Omega_red @ uc / (4 pi^2)``
        (``Omega_red`` the full antisymmetric dim x dim matrix, ``uc`` the lattice vectors as rows).  Not defined for k.p
        models or dim < 2 (:class:`TbkError`)."""
        convention = _check_convention(convention)
        degen_tol = _check_degen_tol(degen_tol)
        k_array, single_point = _normalise_k(k, self.dim)
        n_k = k_array.shape[0]
        n_pairs = self.dim * (self.dim - 1) // 2
        w = np.empty((n_k, self.size), dtype=np.float64)
        curv = np.empty((n_k, self.size, n_pairs), dtype=np.float64)
        _capi.check(
            self._lib.tbk_berry_curvature_host(
                self._handle, k_array.ctypes.data_as(C.c_void_p), n_k, convention, degen_tol,
                w.ctypes.data_as(C.c_void_p), curv.ctypes.data_as(C.c_void_p),
            )
        )
        if single_point:
            return w[0], curv[0]
        return w, curv

    def berry_curvature_device(self, k_dev, convention=2, degen_tol=1e-8, out_w=None, out_c=None):
        """Device-buffer form of :meth:`berry_curvature`: float64 ``[n_k, dim]`` CUDA tensor -> ``(w [n_k, N],
        curv [n_k, N, P])`` float64 tensors, asynchronous on torch's current stream."""
        import torch

        convention = _check_convention(convention)
        degen_tol = _check_degen_tol(degen_tol)
        k_dev = self._check_k_dev(k_dev)
        n_k = k_dev.shape[0]
        n_pairs = self.dim * (self.dim - 1) // 2
        if out_w is None:
            out_w = torch.empty((n_k, self.size), dtype=torch.float64, device=k_dev.device)
        if out_c is None:
            out_c = torch.empty((n_k, self.size, n_pairs), dtype=torch.float64, device=k_dev.device)
        if (tuple(out_w.shape) != (n_k, self.size) or out_w.dtype != torch.float64 or not out_w.is_contiguous()
                or tuple(out_c.shape) != (n_k, self.size, n_pairs) or out_c.dtype != torch.float64
                or not out_c.is_contiguous()):
            raise ValueError("out_w / out_c must be contiguous float64 [n_k, N] / [n_k, N, dim (dim - 1) / 2] tensors")
        _capi.check(
            self._lib.tbk_berry_curvature(
                self._handle, C.c_void_p(k_dev.data_ptr()), n_k, convention, degen_tol, C.c_void_p(out_w.data_ptr()),
                C.c_void_p(out_c.data_ptr()), self._stream(),
            )
        )
        return out_w, out_c

    # ------------------------------------------------------------------ k.p expansion (Model.construct_kdotp)
    def kdotp_coefficients(self, k, order: int):
        """Taylor coefficients of ``Model.construct_kdotp(k, order)`` (reference src/tbmodels/_tb_model.py:942-982).

        Returns ``(powers, coeff)``: the power tuples in the reference's dict order
        (``itertools.product(range(order + 1), repeat=dim)`` filtered by ``sum <= order``) as int32 ``[n_terms, dim]`` and
        the matrices as complex128 ``[n_terms, N, N]`` -- or ``[n_k, n_terms, N, N]`` when ``k`` is a list of expansion
        points (a batched extension; the reference takes a single point)."""
        if order < 0:
            raise ValueError("The order for the k.p model must be positive.")
        k_array, single_point = _normalise_k(k, self.dim)
        powers = np.ascontiguousarray(kdotp_powers(self.dim, int(order)))
        n_k, n_terms = k_array.shape[0], powers.shape[0]
        out = np.empty((n_k, n_terms, self.size, self.size), dtype=np.complex128)
        _capi.check(
            self._lib.tbk_kdotp_coefficients_host(
                self._handle, k_array.ctypes.data_as(C.c_void_p), n_k, powers.ctypes.data_as(C.c_void_p), n_terms,
                out.ctypes.data_as(C.c_void_p),
            )
        )
        return powers, (out[0] if single_point else out)

    def construct_kdotp(self, k, order: int) -> dict:
        """``{power tuple: matrix}`` -- the ``taylor_coefficients`` argument of ``KdotpModel`` -- for ONE expansion point."""
        k_array, single_point = _normalise_k(k, self.dim)
        if not single_point:
            raise ValueError("construct_kdotp expands around a single k-point")
        powers, coeff = self.kdotp_coefficients(k_array[0], order)
        return {tuple(int(x) for x in p): coeff[i] for i, p in enumerate(powers)}

    def kdotp_coefficients_device(self, k_dev, order: int, out=None):
        """Device-buffer form: ``[n_k, dim]`` float64 CUDA tensor -> ``(powers, [n_k, n_terms, N, N] complex128 tensor)``."""
        import torch

        if order < 0:
            raise ValueError("The order for the k.p model must be positive.")
        k_dev = self._check_k_dev(k_dev)
        powers = np.ascontiguousarray(kdotp_powers(self.dim, int(order)))
        shape = (k_dev.shape[0], powers.shape[0], self.size, self.size)
        if out is None:
            out = torch.empty(shape, dtype=torch.complex128, device=k_dev.device)
        elif tuple(out.shape) != shape or out.dtype != torch.complex128 or not out.is_contiguous():
            raise ValueError("out must be a contiguous complex128 tensor [n_k, n_terms, N, N]")
        _capi.check(
            self._lib.tbk_kdotp_coefficients(
                self._handle, C.c_void_p(k_dev.data_ptr()), shape[0], powers.ctypes.data_as(C.c_void_p), shape[1],
                C.c_void_p(out.data_ptr()), self._stream(),
            )
        )
        return powers, out

    # ------------------------------------------------------------------ device buffers (torch tensors as allocators)
    def _stream(self):
        import torch

        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _check_k_dev(self, k_dev):
        import torch

        if not (isinstance(k_dev, torch.Tensor) and k_dev.is_cuda):
            raise TypeError("k_dev must be a CUDA torch.Tensor")
        if k_dev.device.index != self.device:
            raise ValueError(f"k_dev lives on {k_dev.device}, the evaluator on cuda:{self.device}")
        if k_dev.dtype != torch.float64 or k_dev.ndim != 2 or k_dev.shape[1] != self.dim:
            raise ValueError(f"k_dev must be float64 [n_k, {self.dim}]")
        return k_dev.contiguous()

    def hamilton_device(self, k_dev, convention=2, out=None):
        """``[n_k, dim]`` float64 CUDA tensor -> ``[n_k, N, N]`` complex128 CUDA tensor, asynchronous."""
        import torch

        _check_convention(convention)
        k_dev = self._check_k_dev(k_dev)
        n_k = k_dev.shape[0]
        if out is None:
            out = torch.empty((n_k, self.size, self.size), dtype=torch.complex128, device=k_dev.device)
        elif tuple(out.shape) != (n_k, self.size, self.size) or out.dtype != torch.complex128 or not out.is_contiguous():
            raise ValueError("out must be a contiguous complex128 tensor [n_k, N, N]")
        _capi.check(
            self._lib.tbk_hamilton(
                self._handle, C.c_void_p(k_dev.data_ptr()), n_k, int(convention), C.c_void_p(out.data_ptr()),
                self._stream(),
            )
        )
        return out

    def eigenval_device(self, k_dev, out=None):
        """``[n_k, dim]`` float64 CUDA tensor -> ``[n_k, N]`` float64 CUDA tensor (ascending), asynchronous."""
        import torch

        k_dev = self._check_k_dev(k_dev)
        n_k = k_dev.shape[0]
        if out is None:
            out = torch.empty((n_k, self.size), dtype=torch.float64, device=k_dev.device)
        elif tuple(out.shape) != (n_k, self.size) or out.dtype != torch.float64 or not out.is_contiguous():
            raise ValueError("out must be a contiguous float64 tensor [n_k, N]")
        _capi.check(
            self._lib.tbk_eigenval(
                self._handle, C.c_void_p(k_dev.data_ptr()), n_k, C.c_void_p(out.data_ptr()), self._stream()
            )
        )
        return out


def _eigenval_push(self, k_dev, out, peer_ptrs, row_offset):
    """``eigenval_device`` whose chunks are also stored into the peers' result buffers (``tbk_eigenval_push``)."""
    k_dev = self._check_k_dev(k_dev)
    n_k = k_dev.shape[0]
    import torch

    if tuple(out.shape) != (n_k, self.size) or out.dtype != torch.float64 or not out.is_contiguous():
        raise ValueError("out must be a contiguous float64 tensor [n_k, N]")
    arr = (C.c_void_p * max(len(peer_ptrs), 1))(*[C.c_void_p(int(p)) for p in peer_ptrs])
    _capi.check(
        self._lib.tbk_eigenval_push(
            self._handle, C.c_void_p(k_dev.data_ptr()), n_k, C.c_void_p(out.data_ptr()), arr, len(peer_ptrs),
            int(row_offset), self._stream(),
        )
    )
    return out


Evaluator.eigenval_push_device = _eigenval_push


def _default_device() -> int:
    """LOCAL_RANK under torchrun (one process per GPU), else device 0."""
    import os

    try:
        return int(os.environ.get("TBK_DEVICE", os.environ.get("LOCAL_RANK", "0")))
    except ValueError:
        return 0


def fp64_peaks(iters: int = 4000) -> dict:
    """Measured FP64 peaks of the current device in TFLOP/s: ``{"dmma": .., "dfma": ..}``."""
    lib = _capi.load()
    out = {}
    for name, kind in (("dmma", 0), ("dfma", 1), ("dmma+dfma", 2)):
        v = float(lib.tbk_measure_fp64_peak(kind, iters))
        if v < 0:
            raise _capi.TbkError(_capi.TBK_E_CUDA, "FP64 peak micro-benchmark failed (no CUDA device?)")
        out[name] = v
    return out


def int8_peak(iters: int = 1 << 20) -> float:
    """Measured INT8 tensor-core peak of the current device in TOP/s (tcgen05 kind::i8, ``iters`` MMAs per SM)."""
    v = float(_capi.load().tbk_measure_int8_peak(iters))
    if v < 0:
        raise _capi.TbkError(_capi.TBK_E_CUDA, "INT8 peak micro-benchmark failed (no CUDA device?)")
    return v
