"""tbmodels_b200 -- B200-native evaluator for the TBmodels k-space hot path.

Scope (SURVEY.md section 8): ``Model.hamilton(k, convention)`` and ``Model.eigenval(k)`` of
Z2PackDev/TBmodels (reference src/tbmodels/_tb_model.py:1076-1150), evaluated by hand-written sm_100a CUDA
kernels behind the C ABI in ``include/tbk.h``.  Model construction, file formats and model algebra remain
the reference's Python.

Public surface
    pack_model / pack_arrays / PackedModel   host-side packing of ``hop`` / ``pos``
    Evaluator                                owns the device copy; host- and device-buffer entry points
    KModel                                   minimal ``Model`` duck-type (hop, pos, size, dim + the two methods)
    KdotpModel                               ``tbmodels.kdotp.KdotpModel`` duck-type (k.p models, same kernels)
    install / uninstall                      switch ``tbmodels.Model`` itself over to the GPU path
    sharded                                  one-process-per-GPU k-point sharding (torch.distributed)
    io                                       HDF5 model / k-point / eigenvalue files of the `tbmodels eigenvals` CLI
                                             (no h5py needed); `python -m tbmodels_b200 eigenvals` is that command
"""
from . import io  # noqa: F401
from ._capi import TbkError  # noqa: F401
from ._evaluator import Evaluator, fp64_peaks, int8_peak, pinned_empty  # noqa: F401
from ._kdotp import KdotpModel, pack_kdotp  # noqa: F401
from ._model import KModel, SupercellKModel  # noqa: F401
from ._pack import PackedModel, hop_dict, pack_arrays, pack_model  # noqa: F401
from ._patch import evaluator_for, install, install_kdotp, uninstall  # noqa: F401

__version__ = "0.1.0"
