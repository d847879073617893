"""CPU tier: the drop-in boundary of SURVEY 8(b) -- quimb's composed-driver
registration, its partial-eigensolver backend table and the array-level
mirrors of the reference's contraction, split, MPS, DMRG, TEBD, boundary and
compressed-contraction drivers -- checked against what the unmodified
reference computes on numpy.

The reference's values, the inputs it ran on and the names of its
registration points are stored in ``tests/golden/dropin.*``
(``oracle/make_golden.py dropin_cases``), so no quimb is needed here.  The
kernel-launching ABI calls are served by tests/abi_emulator.py (no device
here), so this checks names, signatures, the Array protocol and option
plumbing -- not the CUDA kernels, which the ``-m gpu`` tier covers."""

import sys
import types
import warnings

import numpy as np
import pytest

from tests.conftest import load_golden


@pytest.fixture(scope="module")
def golden():
    return load_golden("dropin")


@pytest.fixture
def qb():
    import quimb_b200
    from tests.abi_emulator import emulated_abi
    with emulated_abi():
        yield quimb_b200


class _Composed:
    """Stand-in for one of quimb's composed functions: records the
    implementation registered for each backend name."""

    def __init__(self):
        self.impls = {}

    def register(self, backend):
        def deco(fn):
            self.impls[backend] = fn
            return fn
        return deco


def test_registration_covers_the_composed_drivers(qb, golden, monkeypatch):
    """register_with_quimb() against stand-ins with exactly the registration
    points the reference offers (its composed functions, the singular-value
    driver table and the partial-eigensolver table)."""
    _, meta = golden
    reg = meta["registrable"]
    decomp = types.ModuleType("quimb.tensor.decomp")
    array_ops = types.ModuleType("quimb.tensor.array_ops")
    for mod, names in ((decomp, reg["decomp"]), (array_ops, reg["array_ops"])):
        for nm in names:
            setattr(mod, nm, _Composed())
    host_svals = {m: (lambda x, *a, _m=m, **kw: ("host", _m)) for m in reg["split_values"]}
    decomp._SPLIT_VALUES_FNS = dict(host_svals)
    base_linalg = types.ModuleType("quimb.linalg.base_linalg")
    base_linalg._EIGS_METHODS = {m: None for m in reg["eigs_methods"]}
    autoray = types.ModuleType("autoray")
    ar_registered = {}
    autoray.register_function = lambda backend, name, fn: ar_registered.__setitem__(
        (backend, name), fn)
    quimb = types.ModuleType("quimb")
    quimb.tensor = types.ModuleType("quimb.tensor")
    quimb.tensor.decomp, quimb.tensor.array_ops = decomp, array_ops
    quimb.linalg = types.ModuleType("quimb.linalg")
    quimb.linalg.base_linalg = base_linalg
    for name, mod in (("autoray", autoray), ("quimb", quimb), ("quimb.tensor", quimb.tensor),
                      ("quimb.tensor.decomp", decomp), ("quimb.tensor.array_ops", array_ops),
                      ("quimb.linalg", quimb.linalg), ("quimb.linalg.base_linalg", base_linalg)):
        monkeypatch.setitem(sys.modules, name, mod)

    names = qb.register_with_quimb()
    for nm in ("svd_truncated", "qr_stabilized", "svd_via_eig_truncated", "eigh_truncated",
               "cholesky_regularized", "polar_right", "polar_left", "fuse", "unfuse",
               "norm_fro", "eigs:QUIMB_B200"):
        assert nm in names
    for nm in names:
        if hasattr(decomp, nm):
            assert "quimb_b200" in getattr(decomp, nm).impls, nm
        elif hasattr(array_ops, nm):
            assert "quimb_b200" in getattr(array_ops, nm).impls, nm
    assert ("quimb_b200", "to_numpy") in ar_registered
    assert base_linalg._EIGS_METHODS["QUIMB_B200"] is qb.integration.eigs_quimb_b200
    # the singular-value drivers: device arrays take the device route, host
    # arrays still reach the reference's own function
    x = np.random.default_rng(3).standard_normal((5, 4))
    for method in ("svd", "svd:eig"):
        fn = decomp._SPLIT_VALUES_FNS[method]
        assert fn(x) == ("host", method)
        s = fn(qb.asarray(x))
        assert isinstance(s, qb.Array)
        np.testing.assert_allclose(np.sort(s.to_numpy())[::-1],
                                   np.linalg.svd(x, compute_uv=False), atol=1e-12)


def test_tensor_contract_and_matmul_stay_on_the_backend(qb, golden):
    """``Tensor @``, ``tensor_contract`` with explicit / hyper output indices and
    a complex full contraction with the mantissa / exponent split, against the
    reference's numpy results."""
    data, meta = golden
    inds = meta["contract_inds"]
    dev = {k: qb.asarray(data[f"contract__{k}"]) for k in inds}

    def contract(keys, **kw):
        return qb.tensor_contract([dev[k] for k in keys], [inds[k] for k in keys], **kw)

    out, out_inds = contract("ab")
    assert isinstance(out, qb.Array) and tuple(out_inds) == tuple(meta["contract_ab_inds"])
    np.testing.assert_allclose(out.to_numpy(), data["contract__ab"], atol=1e-13)
    out3, _ = contract("abc", output_inds="ea")
    assert isinstance(out3, qb.Array)
    np.testing.assert_allclose(out3.to_numpy(), data["contract__abc_ea"], atol=1e-13)
    outh, _ = contract(("h1", "h2", "h3"), output_inds="xyz")
    np.testing.assert_allclose(outh.to_numpy(), data["contract__hyper_xyz"], atol=1e-13)
    refz = complex(*meta["contract_z"])
    outz, _ = contract(("z1", "z2"))
    assert abs(complex(outz.to_numpy().reshape(())) - refz) < 1e-13
    (m, e), _ = contract(("z1", "z2"), strip_exponent=True)
    strip = meta["contract_z_strip"]
    assert abs(complex(m.to_numpy().reshape(())) - complex(*strip["mantissa"])) < 1e-12
    assert e == pytest.approx(strip["exponent"], abs=1e-12)
    assert abs(complex(m.to_numpy().reshape(())) * 10 ** e - refz) < 1e-12


@pytest.mark.parametrize("method,kw", [
    ("svd", dict(cutoff=1e-3, cutoff_mode="rel")), ("svd", dict(max_bond=3, absorb="left")),
    ("svd:eig", dict(max_bond=4)), ("qr", {}), ("lq", {}), ("eigh", dict(max_bond=4)),
    ("polar_right", {}), ("polar_left", {}),
])
def test_tensor_split_methods_through_quimb(qb, golden, method, kw):
    """``Tensor.split(..., get='arrays')`` of the reference, mirrored by
    ``tensor_split``: same factor shapes, same product of the factors (the
    gauge-free comparison)."""
    data, meta = golden
    (k, case), = [(k, c) for k, c in enumerate(meta["splits"])
                  if c["method"] == method and c["kw"] == kw]
    x = data[f"split{k}__x"]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        out = qb.tensor_split(qb.asarray(x), case["inds"], case["left_inds"],
                              method=method, **kw)
    assert all(isinstance(o, qb.Array) for o in out)
    assert [list(o.shape) for o in out] == case["shapes"]
    prod_out = np.tensordot(out[0].to_numpy(), out[-1].to_numpy(), 1)
    np.testing.assert_allclose(prod_out, data[f"split{k}__product"], atol=1e-10)


def _fresh(data, key, n):
    from quimb_b200 import mps
    return [mps.site_lpr(data[f"{key}__{i}"], "lrp", i, n) for i in range(n)]


def _dense(sites):
    from oracle import dmrg_np as dm
    return dm.mps_to_dense([np.asarray(s.to_numpy()) for s in sites]).reshape(-1)


def _mpo(data, key, n):
    return [data[f"{key}__{i}"] for i in range(n)]


def test_canonize_compress_and_linear_operator(qb, golden):
    """MPS left_canonize / compress / expec_TN_1D and TNLinearOperator of the
    reference, mirrored on device arrays."""
    from quimb_b200 import tebd as tb
    data, meta = golden
    c = meta["canon"]
    p = _fresh(data, "canon_p", 6)
    assert abs(complex(tb.mps_overlap(p, p)) - c["norm0"]) < 1e-12
    tb.left_canonize(p)
    assert all(isinstance(a, qb.Array) for a in p)
    assert abs(complex(tb.mps_overlap(p, p)) - c["norm_canon"]) < 1e-12
    tb.mps_compress(p, max_bond=3)
    assert max(a.shape[2] for a in p[:-1]) == c["max_bond"] == 3
    assert abs(complex(tb.mps_overlap(p, p)) - c["norm_compressed"]) < 1e-10
    e = qb.mps_expec(p, _mpo(data, "heis6", 6), shape="lpr", mpo_shape="lrud")
    assert abs(float(e.to_numpy().real) - c["expec"]) < 1e-10
    # TNLinearOperator: device matvec of a host vector, and its dense form
    arrays = [qb.asarray(data[f"linop__t{k}"]) for k in range(2)]
    A = qb.TNLinearOperator(arrays, [("a", "w", "b"), ("w", "p", "q")], ("a", "p"), ("b", "q"))
    v = qb.asarray(data["linop__v"])
    out = A.matvec(v)                        # device in, device out
    assert isinstance(out, qb.Array)
    np.testing.assert_allclose(out.to_numpy(), data["linop__matvec"], atol=1e-12)
    np.testing.assert_allclose(A.to_dense().to_numpy(), data["linop__dense"], atol=1e-12)


def test_reference_dmrg2_default_eigensolver_path(qb, golden):
    """quimb's default local eigensolve hands the effective Hamiltonian to
    scipy ARPACK on the host (dmrg.py:626-645); the mirror's parity mode does
    the same with device products: same energy as the reference's run."""
    data, meta = golden
    d = qb.DMRG2.from_quimb_layout(_mpo(data, "heis8", 8), [8, 16, 32], cutoffs=1e-10,
                                   p0_arrays=[data[f"dmrg_p4__{i}"] for i in range(8)])
    d.opts["local_eig_backend"] = "SCIPY"
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        d.solve(tol=1e-8, max_sweeps=5)
    assert abs(float(d.energy) - meta["dmrg"]["default_energy"]) < 1e-6


@pytest.mark.parametrize("dense", [True, False])
def test_reference_dmrg2_runs_on_device_arrays(qb, golden, dense):
    """DMRG2 with the device eigensolver against the reference's runs: energy,
    exact ground state, bond sizes.  The mirror has no dense local-eigensolve
    option, so ``dense`` only selects which reference run (quimb's
    ``local_eig_ham_dense`` set to it) the same device computation is
    compared with."""
    data, meta = golden
    ref = meta["dmrg"][f"dense_{dense}"]
    L = 8
    d = qb.DMRG2.from_quimb_layout(_mpo(data, "heis8", L), [8, 16], cutoffs=1e-10,
                                   p0_arrays=[data[f"dmrg_p8__{i}"] for i in range(L)])
    d.solve(tol=1e-9, max_sweeps=5)
    assert all(isinstance(a, qb.Array) for a in d.state)
    assert abs(float(d.energy) - ref["energy"]) < 1e-6
    assert abs(float(d.energy) - meta["dmrg"]["exact"]) < 1e-6
    assert [a.shape[2] for a in d.state[:-1]] == ref["bonds"]


def test_reference_callers_either_side_of_the_path(qb, golden):
    """The drivers around the hot path (SURVEY 8f: boundary contraction,
    circuits, TEBD, DMRG1, MPS gates / arithmetic) on device arrays, against
    the reference's numpy runs."""
    from quimb_b200 import boundary as bd, tebd as tb
    data, meta = golden
    cl = meta["callers"]
    # PEPS norm by boundary-MPS contraction (tn2d/core.py:2528-2543)
    arrays = [[data[f"peps__{i}_{j}"] for j in range(4)] for i in range(4)]
    ts, Lx, Ly = bd.peps_norm_tensors(arrays)
    v = bd.contract_boundary(ts, Lx, Ly, max_bond=8, cutoff=0.0, layer_tags=("KET", "BRA"))
    ref = complex(*cl["peps_norm"])
    assert abs(complex(v) - ref) < 1e-10 * abs(ref)
    ising = [(data[f"ising__t{k}"], r["inds"], tuple(r["site"]), r["layer"])
             for k, r in enumerate(cl["ising_tensors"])]
    assert abs(float(np.real(bd.contract_boundary(ising, 4, 4, max_bond=8)))
               - cl["ising_Z"]) < 1e-6

    # circuit amplitudes (circuit/exact.py:90-98): the unsimplified amplitude
    # networks (initial states, gates, projections) contracted on the backend
    for bits in ("01001", "00000"):
        inds = cl[f"amp_{bits}_inds"]
        assert len(inds) > 20
        arrays = [qb.asarray(data[f"amp_{bits}__t{k}"]) for k in range(len(inds))]
        out, _ = qb.tensor_contract(arrays, inds, output_inds=())
        assert abs(complex(out.to_numpy().reshape(())) - complex(*cl[f"amp_{bits}"])) < 1e-12

    # TEBD from the Neel state (tn1d/tebd.py)
    H = tb.LocalHam1D(6, H2=data["tebd__h2"])
    p0 = [np.zeros((1, 2, 1)) for _ in range(6)]
    for i in range(6):
        p0[i][0, i % 2, 0] = 1.0
    t = tb.TEBD(p0, H)
    t.update_to(0.2, dt=0.05, order=2)
    assert isinstance(t.pt[2], qb.Array)
    ref = data["tebd__dense"]
    assert abs(abs(np.vdot(ref, _dense(t.pt))) - abs(np.vdot(ref, ref))) < 1e-10

    # DMRG1 with the device eigensolver
    d = qb.DMRG1.from_quimb_layout(_mpo(data, "heis8", 8), [8, 16],
                                   p0_arrays=[data[f"dmrg_p8__{i}"] for i in range(8)])
    d.solve(tol=1e-8, max_sweeps=4)
    assert abs(float(d.energy) - meta["dmrg"]["dmrg1_energy"]) < 1e-7

    # MPS gates, MPO application, addition, entropy
    G = qb.asarray(data["gates__G"])
    for where, fn in (((2, 3), tb.gate_split), ((0, 4), tb.gate_with_auto_swap)):
        # the reference promotes a real state to the gate's complex dtype
        p = [a.astype(G.dtype) for a in _fresh(data, "gates_p", 6)]
        fn(p, G, where, cutoff=1e-12)
        np.testing.assert_allclose(_dense(p), data[f"gates__{fn.__name__}"], atol=1e-10)
    p = _fresh(data, "gates_p", 6)
    q = _fresh(data, "gates_q", 6)
    Hp = tb.mpo_apply(_mpo(data, "heis6", 6), p, mpo_shape="lrud")
    np.testing.assert_allclose(_dense(Hp), data["gates__apply"], atol=1e-10)
    np.testing.assert_allclose(_dense(tb.mps_add(p, q)), data["gates__add"], atol=1e-12)
    # entropy of the first three sites: Schmidt values at the bond (2, 3)
    tb.canonicalize(p, 2)
    a = p[2]
    s = qb.split.svdvals(a.reshape(a.shape[0] * a.shape[1], a.shape[2])).to_numpy()
    s2 = s[s > 0] ** 2
    assert abs(float(-np.sum(s2 * np.log2(s2))) - cl["entropy3"]) < 1e-10


def test_reference_compressed_contraction_runs_on_the_backend_and_matches_the_mirror(qb, golden):
    """The reference's ``_contract_compressed_tid_sequence`` ('basic' mode,
    tensor_core.py:8560-8780) against ``contract_compressed`` on the same
    sequence, with a bond limit that truncates: the stored values differ from
    the exact contraction, and from each other through ``compress_late``."""
    data, meta = golden
    m = meta["compressed"]
    values = [r["value"] for r in m["runs"]]
    assert min(abs(v - m["exact"]) for v in values) > 1e-3 * abs(m["exact"])
    assert abs(values[0] - values[1]) > 1e-3 * abs(m["exact"])
    arrays = [qb.asarray(data[f"compressed__t{k}"]) for k in range(len(m["inputs"]))]
    inputs = [tuple(i) for i in m["inputs"]]
    seq = [tuple(p) for p in m["seq"]]
    for run in m["runs"]:
        kw = {k: v for k, v in run["kw"].items() if k not in ("tree_gauge_distance", "compress_mode")}
        out = qb.contract_compressed(arrays, inputs, (), seq, **kw)
        assert abs(out.item() - run["value"]) <= 1e-9 * abs(run["value"]), run["kw"]
