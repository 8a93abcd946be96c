"""``tbmodels_b200.install()`` on the reference's ``tbmodels.Model`` class, on a B200.

With the unmodified reference importable (``oracle/ref_shim.py``: a TBmodels source tree, or the verified archive
``oracle/build_ref.py`` keeps under ``oracle/_ref``), these tests patch the real class.  Without it they patch
``oracle/ref_standin.py``: the same data layout (half-set ``hop`` dict, csr matrices when ``sparse=True``) with the oracle's
numpy methods, which tests/test_oracle_golden.py pins against stored outputs of the unmodified reference.  Either way they
run the bodies of the reference's own ``tests/test_hamilton.py:21-42`` and ``tests/test_eigenval.py:17-20`` (dense and
``sparse=True``, ``tests/conftest.py:155-206``) against the installed GPU methods, with every warning raised as an error
around our calls (reference ``pytest.ini:3``).  They compare with the class's own numpy methods at the north_star bounds
and with the reference's regression data for the same models (``tests/golden/ref_regression.npz``).
"""
import itertools
import pickle
import warnings
from collections import ChainMap

import numpy as np
import pytest
from numpy.testing import assert_allclose

from conftest import assert_eig_close, load_golden

pytestmark = pytest.mark.gpu

# reference tests/parameters.py
T_VALUES = [(t1, t2) for t1 in [-0.1, 0.2, 0.3] for t2 in [-0.2, 0.5]]
KPT = [(0.1, 0.2, 0.7), (-0.3, 0.5, 0.2), (0.0, 0.0, 0.0), (0.1, -0.9, -0.7)]


@pytest.fixture(scope="module")
def ref():
    from conftest import gpu_available

    if not gpu_available():
        pytest.skip("no CUDA device")
    from oracle import ref_shim

    import tbmodels_b200 as tbk

    if ref_shim.reference_available():
        tb = ref_shim.import_reference()
    else:
        from oracle import ref_standin as tb
    orig = (tb.Model.hamilton, tb.Model.eigenval, tb.kdotp.KdotpModel.hamilton, tb.kdotp.KdotpModel.eigenval,
            tb.Model.construct_kdotp)
    if tb.__name__ == "tbmodels":
        tbk.install()
    else:
        tbk.install(tb.Model)
        tbk.install_kdotp(tb.kdotp.KdotpModel)
    assert tb.Model.hamilton is not orig[0] and tb.Model.eigenval is not orig[1] and tb.Model.construct_kdotp is not orig[4]
    assert tb.kdotp.KdotpModel.hamilton is not orig[2] and tb.kdotp.KdotpModel.eigenval is not orig[3]
    yield tb, orig
    tbk.uninstall()
    assert tb.Model.hamilton is orig[0] and tb.Model.eigenval is orig[1] and tb.Model.construct_kdotp is orig[4]
    assert tb.kdotp.KdotpModel.hamilton is orig[2] and tb.kdotp.KdotpModel.eigenval is orig[3]


def ref_regression(t_values):
    """The reference's regression data (its tests/regression_data/test_hamilton|test_eigenval) for ``get_model(*t_values)``
    at ``KPT``: the stored arrays and the index of ``t_values`` in them."""
    d = load_golden("ref_regression.npz")
    assert np.array_equal(d["kpt"], np.array(KPT))
    return d, [tuple(t) for t in d["t_values"].tolist()].index(tuple(t_values))


def get_model(tb, t1, t2, sparse, **kwargs):
    """Reference tests/conftest.py:155-189 (``get_model_clean``), restated: the test fixture of the reference suite."""
    dim = kwargs.get("dim", 3)
    defaults = {"pos": [[0] * 2, [0.5] * 2], "occ": 1, "on_site": (1, -1), "size": 2, "dim": None, "sparse": sparse}
    for position in defaults["pos"]:
        position.extend([0] * (dim - 2))
    with warnings.catch_warnings():  # the reference's own construction code warns under numpy 2 (sparse __array__)
        warnings.simplefilter("ignore")
        model = tb.Model(**ChainMap(kwargs, defaults))
        for phase, r_part in zip([1, -1j, 1j, -1], itertools.product([0, -1], [0, -1])):
            model.add_hop(t1 * phase, 0, 1, list(r_part) + [0] * (dim - 2))
        for r_part in itertools.permutations([0, 1]):
            R = list(r_part) + [0] * (dim - 2)
            model.add_hop(t2, 0, 0, R)
            model.add_hop(-t2, 1, 1, R)
    return model


class strict:
    """Every warning raised inside the block is an error (reference pytest.ini: ``filterwarnings = error``)."""

    def __enter__(self):
        self._cm = warnings.catch_warnings()
        self._cm.__enter__()
        warnings.simplefilter("error")
        warnings.simplefilter("ignore", ImportWarning)

    def __exit__(self, *exc):
        return self._cm.__exit__(*exc)


@pytest.mark.parametrize("sparse", [True, False])
@pytest.mark.parametrize("convention", [1, 2])
@pytest.mark.parametrize("t_values", T_VALUES)
def test_parallel_hamilton(ref, t_values, convention, sparse):
    """reference tests/test_hamilton.py:21-32 on the GPU methods + parity with the reference's numpy ``hamilton``."""
    tb, orig = ref
    model = get_model(tb, *t_values, sparse=sparse)
    with strict():
        batched = model.hamilton(KPT, convention=convention)
        single = [model.hamilton(k, convention=convention) for k in KPT]
    assert_allclose(batched, single)
    assert isinstance(batched, np.ndarray) and batched.shape == (len(KPT), 2, 2) and batched.dtype == np.complex128
    assert single[0].shape == (2, 2)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        want = orig[0](model, KPT, convention=convention)
    scale = max(abs(t_values[0]), abs(t_values[1]), 1.0)
    assert np.abs(batched - want).max() <= 1e-11 * scale
    d, ti = ref_regression(t_values)
    assert np.abs(batched - np.array([d[f"H{convention}_t{ti}_k{ki}"] for ki in range(len(KPT))])).max() <= 1e-11 * scale


@pytest.mark.parametrize("convention", ["a", "1", None])
def test_invalid_convention(ref, convention):
    """reference tests/test_hamilton.py:35-42."""
    tb, _ = ref
    model = get_model(tb, 0, 0.1, sparse=False)
    with pytest.raises(ValueError):
        model.hamilton((0, 0, 0), convention=convention)


@pytest.mark.parametrize("sparse", [True, False])
@pytest.mark.parametrize("t_values", T_VALUES)
def test_parallel_eigenval(ref, t_values, sparse):
    """reference tests/test_eigenval.py:17-20 + return types (:1148-1150) + parity with the reference's ``eigenval``."""
    tb, orig = ref
    model = get_model(tb, *t_values, sparse=sparse)
    with strict():
        batched = model.eigenval(KPT)
        single = [model.eigenval(k) for k in KPT]
    assert_allclose(batched, single)
    assert isinstance(batched, list) and len(batched) == len(KPT) and all(e.shape == (2,) for e in batched)
    assert isinstance(single[0], np.ndarray) and single[0].shape == (2,)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        want = orig[1](model, KPT)
    assert_eig_close(np.array(batched), np.array(want), f"Model sparse={sparse}")
    d, ti = ref_regression(t_values)
    assert_eig_close(np.array(batched), np.array([d[f"E_t{ti}_k{ki}"] for ki in range(len(KPT))]), "regression data")


@pytest.mark.parametrize("sparse", [True, False])
def test_silicon_known_answer_and_cli_handoff(ref, sparse):
    """The silicon Wannier model as a real ``tbmodels.Model``: ``model.eigenval`` handed over as a bare callable the way
    ``tbmodels eigenvals`` does (reference src/tbmodels/_cli.py:255-257) reproduces the reference's own known answer
    (tests/samples/cli_eigenvals/silicon_eigenvals.hdf5, atol 1e-10 as in tests/test_cli_eigenvals.py:47-50)."""
    tb, _ = ref
    d = known = load_golden("silicon_cli_eigenvals.npz")  # model of tests/samples/cli_eigenvals + its known answer
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model = tb.Model(hop={tuple(int(x) for x in R): m for R, m in zip(d["R"], d["hop"])}, size=d["pos"].shape[0], dim=3,
                         pos=d["pos"], contains_cc=False, sparse=sparse)
    eigenval_function = model.eigenval
    with strict():
        got = np.array(eigenval_function(known["k"]))
    assert np.abs(got - known["eig"]).max() <= 1e-10
    # the instance carries no device state: pickling works and the copy evaluates to the same bits
    assert not any("tbk" in key or "evaluator" in key.lower() for key in model.__dict__)
    clone = pickle.loads(pickle.dumps(model))
    assert np.array_equal(np.array(clone.eigenval(known["k"])), got)


def test_mutation_and_model_algebra(ref):
    """In-place ``add_hop`` (reference :1196-1215) invalidates the cached device copy; models derived by the reference's
    own algebra (``supercell`` :1645-1724, arithmetic :2030-2118) evaluate on the GPU like any other."""
    tb, orig = ref
    model = get_model(tb, 0.3, -0.2, sparse=False)
    k = np.array(KPT)
    before = np.array(model.eigenval(k))
    model.add_hop(0.25, 0, 1, (1, 0, 1))
    after = np.array(model.eigenval(k))
    assert np.abs(after - before).max() > 1e-3
    assert_eig_close(after, np.array(orig[1](model, k)), "after add_hop")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        big = model.supercell((2, 1, 2))
        summed = model + 0.5 * model
    for m in (big, summed):
        assert_eig_close(np.array(m.eigenval(k)), np.array(orig[1](m, k)), f"derived N={m.size}")
        assert np.abs(m.hamilton(k, convention=1) - orig[0](m, k, convention=1)).max() <= 1e-11


def test_kdotp_model(ref):
    """``Model.construct_kdotp`` (reference :942-982) -> real ``KdotpModel`` -> installed GPU methods (kdotp.py:51-100)."""
    tb, orig = ref
    model = get_model(tb, 0.2, 0.5, sparse=False)
    with strict():
        kp = model.construct_kdotp((0.1, 0.2, 0.3), order=3)  # the installed GPU version
    assert isinstance(kp, tb.kdotp.KdotpModel)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        kp_ref = orig[4](model, (0.1, 0.2, 0.3), order=3)  # the reference's numpy version
    assert list(kp.taylor_coefficients) == list(kp_ref.taylor_coefficients)
    for key, want in kp_ref.taylor_coefficients.items():
        assert np.abs(kp.taylor_coefficients[key] - want).max() <= 1e-11 * (2 * np.pi) ** sum(key)
    with pytest.raises(ValueError):
        model.construct_kdotp((0.1, 0.2, 0.3), order=-1)
    sparse_model = get_model(tb, 0.2, 0.5, sparse=True)
    with strict():
        kp_sparse = sparse_model.construct_kdotp((0.1, 0.2, 0.3), order=2)
    for key, want in kp_sparse.taylor_coefficients.items():
        assert np.array_equal(want, kp.taylor_coefficients[key])
    k = np.array([[0.01, -0.02, 0.03], [0.0, 0.0, 0.0], [0.05, 0.04, -0.01]])
    with strict():
        h = kp.hamilton(k)
        e = kp.eigenval(k)
        e0 = kp.eigenval(k[0])
    want_h = orig[2](kp, k)
    want_e = np.array(orig[3](kp, k))
    assert np.abs(h - want_h).max() <= 1e-11 * max(np.abs(want_h).max(), 1.0)
    assert isinstance(e, list) and e0.shape == (2,)
    assert_eig_close(np.array(e), want_e, "kdotp")
