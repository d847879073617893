"""Generate tests/golden/*.npz by running the UNMODIFIED reference
(/root/reference, quimb @ 97ceeae) on its numpy backend.

The reference's third-party layer (autoray / cotengra / cytoolz) is not
installable offline; oracle/shims provides functional stand-ins that only
route calls -- all arithmetic is the reference's own code (tensor_core,
decomp incl. its numba kernels, dmrg, scipy ARPACK) on numpy.

Run in the build container only:   python oracle/make_golden.py
(the GPU box has no /root/reference; tests read the committed fixtures).
"""

import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get("QUIMB_REFERENCE", "/root/reference")
sys.path.insert(0, os.path.join(HERE, "shims"))
sys.path.insert(0, REF)
sys.path.insert(0, ROOT)

import quimb as qu  # noqa: E402
import quimb.tensor as qtn  # noqa: E402
from quimb.tensor import decomp  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
os.makedirs(OUT, exist_ok=True)


def contract_cases():
    rng = np.random.default_rng(0)
    cases = [
        # (name, [(shape, inds), ...], output_inds or None, dtype)
        ("pair_cfg1", [((6, 5, 4, 3), "abcd"), ((4, 3, 7, 2), "cdef")], None, "float64"),
        ("pair_perm", [((6, 4, 5, 3), "acbd"), ((3, 2, 4, 7), "dfce")], None, "float64"),
        ("outer", [((3, 4), "ab"), ((5,), "c")], None, "float64"),
        ("scalar", [((3, 4, 5), "abc"), ((5, 4, 3), "cba")], None, "float64"),
        ("three", [((3, 4), "ab"), ((4, 5), "bc"), ((5, 6), "cd")], None, "float64"),
        ("env4", [((7, 5, 7), "xwa"), ((7, 2, 6), "apb"), ((5, 4, 2, 2), "wvqp"),
                  ((7, 2, 6), "xqy")], None, "float64"),
        ("hyper_out", [((3, 4), "ab"), ((4, 5), "bc"), ((4, 2), "bd")], "abcd"[0:1] + "cd", "float64"),
        ("batch_keep", [((3, 4), "ab"), ((3, 5), "ac")], "abc", "float64"),
        ("cplx_pair", [((4, 3, 5), "abc"), ((5, 3, 2), "cbd")], None, "complex128"),
        ("cplx_scalar", [((4, 3), "ab"), ((4, 3), "ab")], None, "complex128"),
        ("order_out", [((2, 3, 4), "abc"), ((4, 5), "cd")], "dab", "float64"),
        ("rank0", [((), ""), ((3, 2), "ab")], None, "float64"),
    ]
    store = {}
    meta = {}
    for name, tensors, out_inds, dtype in cases:
        ts = []
        for k, (shape, inds) in enumerate(tensors):
            x = rng.standard_normal(shape)
            if dtype.startswith("complex"):
                x = x + 1j * rng.standard_normal(shape)
            x = np.asarray(x, dtype=dtype)
            store[f"{name}__in{k}"] = x
            ts.append(qtn.Tensor(x, inds=tuple(inds)))
        kw = {} if out_inds is None else {"output_inds": tuple(out_inds)}
        res = qtn.tensor_contract(*ts, preserve_tensor=True, **kw)
        store[f"{name}__out"] = np.asarray(res.data)
        meta[name] = {
            "inds": [list(i) for _, i in tensors],
            "output_inds": None if out_inds is None else list(out_inds),
            "result_inds": list(res.inds),
            "dtype": dtype,
        }
        # strip_exponent (+ a base exponent) through the reference's
        # tensor_contract (tensor_core.py:330-341)
        if name in ("three", "env4", "cplx_pair", "scalar", "order_out"):
            big = [qtn.Tensor(t.data * (10.0 ** (40 * (k + 1))), inds=t.inds)
                   for k, t in enumerate(ts)]
            rs, ex = qtn.tensor_contract(*big, preserve_tensor=True, strip_exponent=True,
                                         exponent=2.5, **kw)
            store[f"{name}__strip_mantissa"] = np.asarray(rs.data)
            meta[name]["strip"] = {"exponent": float(ex), "base_exponent": 2.5,
                                   "input_scales": [40 * (k + 1) for k in range(len(ts))]}
    # error behaviour: index appearing three times without output_inds
    try:
        qtn.tensor_contract(qtn.rand_tensor((2, 2), "ab"), qtn.rand_tensor((2, 2), "bc"),
                            qtn.rand_tensor((2, 2), "bd"))
        meta["_triple_index_error"] = None
    except ValueError as e:
        meta["_triple_index_error"] = str(e)
    np.savez_compressed(os.path.join(OUT, "contract.npz"), **store)
    json.dump(meta, open(os.path.join(OUT, "contract.json"), "w"), indent=1)


def decomp_cases():
    rng = np.random.default_rng(1)
    store, meta = {}, {}
    # known answers restated from the reference's own tests
    s = np.array([3.0, 2.0, 1.0, 0.1])
    meta["svals_to_keep"] = {
        "s": s.tolist(),
        "cases": [
            [c, m, int(decomp._compute_number_svals_to_keep_numba(s, c, m))]
            for c, m in [(1.1, 1), (0.5, 2), (1.02, 3), (0.1, 4), (1.2, 5),
                         (0.2, 6), (1e-12, 3), (100.0, 3), (0.0, 1), (5.0, 6)]
        ],
    }
    mats = {
        "rect_tall": rng.standard_normal((24, 10)),
        "rect_wide": rng.standard_normal((9, 20)),
        "square": rng.standard_normal((16, 16)),
        "lowrank": rng.standard_normal((20, 4)) @ rng.standard_normal((4, 18)),
        "cplx": rng.standard_normal((12, 14)) + 1j * rng.standard_normal((12, 14)),
        "decay": (np.linalg.qr(rng.standard_normal((20, 20)))[0]
                  * (0.5 ** np.arange(20))[None, :])
                 @ np.linalg.qr(rng.standard_normal((20, 20)))[0],
    }
    svd_cases = []
    for mname, x in mats.items():
        store[f"mat__{mname}"] = x
        for (cutoff, mode, max_bond, absorb, renorm) in [
            (-1.0, 4, -1, None, 0),
            (1e-2, 4, -1, 0, 0),
            (1e-3, 3, -1, -1, 0),
            (1e-1, 1, -1, 1, 0),
            (1e-2, 2, 6, 0, 0),
            (-1.0, 4, 5, 1, 0),
            (1e-2, 4, -1, 0, 2),
            (1e-2, 6, -1, 0, 1),
            (0.3, 5, -1, None, 0),
            (0.0, 3, 7, -1, 0),
        ]:
            info = {"error": None}
            left, sv, right = decomp.svd_truncated(
                x, cutoff=cutoff, cutoff_mode=mode, max_bond=max_bond,
                absorb=absorb, renorm=renorm, info=info)
            key = f"svd__{mname}__{len(svd_cases)}"
            if left is not None and right is not None:
                rec = left @ (np.diag(sv) @ right if sv is not None else right)
            else:
                rec = None
            k = (left.shape[1] if left is not None else right.shape[0])
            if sv is not None:
                store[key + "__s"] = sv
            if rec is not None:
                store[key + "__rec"] = rec
            svd_cases.append({
                "key": key, "mat": mname, "cutoff": cutoff, "cutoff_mode": mode,
                "max_bond": max_bond, "absorb": absorb, "renorm": renorm,
                "n_keep": int(k), "error": float(info["error"]),
            })
    meta["svd_cases"] = svd_cases
    qr_cases = []
    for mname in ("rect_tall", "square", "cplx", "rect_wide"):
        x = mats[mname]
        for absorb in (1, 10, 11, -1, -10, -11):
            left, _, right = decomp.qr_stabilized(x.copy(), absorb=absorb)
            key = f"qr__{mname}__{absorb}"
            if left is not None:
                store[key + "__left"] = left
            if right is not None:
                store[key + "__right"] = right
            qr_cases.append({"key": key, "mat": mname, "absorb": absorb})
    meta["qr_cases"] = qr_cases
    # tensor_split through the Tensor interface (transpose + fuse + split + unfuse)
    x = rng.standard_normal((4, 3, 5, 2))
    store["split__x"] = x
    t = qtn.Tensor(x, inds="abcd")
    split_cases = []
    for kw in [
        dict(left_inds="ac", method="svd", cutoff=1e-10, absorb="both"),
        dict(left_inds="ca", right_inds="db", method="svd", max_bond=4, cutoff=0.0, absorb="right"),
        dict(left_inds="b", method="svd", cutoff=1e-1, cutoff_mode="sum2", absorb="left"),
        dict(left_inds="ab", method="qr"),
        dict(left_inds="ab", method="lq"),
        dict(left_inds="d", method="svd", absorb=None, cutoff=0.0),
    ]:
        kw = {k: (tuple(v) if k.endswith("inds") else v) for k, v in kw.items()}
        arrs = t.split(get="arrays", **kw)
        key = f"split__{len(split_cases)}"
        for j, a in enumerate(arrs):
            if a is not None:
                store[f"{key}__{j}"] = np.asarray(a)
        split_cases.append({"key": key, "n_out": len(arrs),
                            "kw": {k: (list(v) if k.endswith("inds") else v)
                                   for k, v in kw.items()}})
    meta["split_cases"] = split_cases
    # bond canonisation / compression through the Tensor interface
    ta = qtn.Tensor(rng.standard_normal((6, 12, 5)), inds=("a", "x", "b"))
    tb = qtn.Tensor(rng.standard_normal((4, 12, 3)), inds=("c", "x", "d"))
    store["bond__a"], store["bond__b"] = ta.data.copy(), tb.data.copy()
    ca, cb = ta.copy(), tb.copy()
    qtn.tensor_canonize_bond(ca, cb, absorb="right")
    store["bond__canon_a"], store["bond__canon_b"] = np.asarray(ca.data), np.asarray(cb.data)
    meta["bond_canon_inds"] = [list(ca.inds), list(cb.inds)]
    bond_cases = []
    for kw in [dict(max_bond=5, cutoff=0.0, absorb="both"), dict(max_bond=None, cutoff=1e-1, absorb="right"),
               dict(max_bond=7, cutoff=1e-10, absorb="left")]:
        xa, xb = ta.copy(), tb.copy()
        qtn.tensor_compress_bond(xa, xb, **kw)
        key = f"bond__cmp{len(bond_cases)}"
        store[key + "_a"], store[key + "_b"] = np.asarray(xa.data), np.asarray(xb.data)
        bond_cases.append({"key": key, "kw": kw, "inds": [list(xa.inds), list(xb.inds)],
                           "bond": int(xa.ind_size("x"))})
    meta["bond_cases"] = bond_cases
    # parse_split_opts codes
    meta["parse_split_opts"] = []
    for kw in [dict(), dict(method="svd", absorb="left", max_bond=7, cutoff=1e-3, cutoff_mode="sum2"),
               dict(method="svd", renorm=True, cutoff_mode="rsum1"), dict(method="qr"),
               dict(method="svd", absorb=None, cutoff=None, max_bond=None)]:
        method, opts = decomp.parse_split_opts(**kw)
        meta["parse_split_opts"].append({"kw": kw, "method": method, "opts": opts})
    np.savez_compressed(os.path.join(OUT, "decomp.npz"), **store)
    json.dump(meta, open(os.path.join(OUT, "decomp.json"), "w"), indent=1, default=str)


def _gauge_free(left, sv, right):
    """Gauge-invariant images of a split result for storage."""
    out = {}
    if sv is not None:
        out["s"] = np.asarray(sv)
    if left is not None and right is not None:
        out["rec"] = left @ (np.diag(sv) @ right if sv is not None else right)
    elif left is not None:
        out["lgram"] = left @ left.conj().T
    elif right is not None:
        out["rgram"] = right.conj().T @ right
    return out


def decomp2_cases():
    """Gram-matrix SVD ('svd:eig'), Hermitian 'eigh' split and randomized SVD
    ('svd:rand') of the reference on its numpy backend."""
    rng = np.random.default_rng(11)
    store, meta = {}, {}
    q1 = np.linalg.qr(rng.standard_normal((20, 20)))[0]
    q2 = np.linalg.qr(rng.standard_normal((20, 20)))[0]
    sym = rng.standard_normal((18, 18))
    hc = rng.standard_normal((14, 14)) + 1j * rng.standard_normal((14, 14))
    ps = rng.standard_normal((16, 9))
    mats = {
        "tall": rng.standard_normal((24, 10)),
        "wide": rng.standard_normal((9, 20)),
        "square": rng.standard_normal((16, 16)),
        "lowrank": rng.standard_normal((20, 4)) @ rng.standard_normal((4, 18)),
        "cplx": rng.standard_normal((12, 14)) + 1j * rng.standard_normal((12, 14)),
        "decay": (q1 * (0.6 ** np.arange(20))[None, :]) @ q2,
        "sym": sym + sym.T,
        "psd": ps @ ps.T,
        "herm": hc + hc.conj().T,
    }
    for k, v in mats.items():
        store[f"mat__{k}"] = v
    eig_cases = []
    for mname in ("tall", "wide", "square", "lowrank", "cplx", "decay"):
        x = mats[mname]
        for (cutoff, mode, max_bond, absorb, renorm, want_err) in [
            (-1.0, 4, -1, None, 0, False),
            (1e-2, 4, -1, 0, 0, True),
            (1e-3, 3, -1, -1, 0, True),
            (-1.0, 4, 5, 1, 0, False),
            (-1.0, 4, 6, -1, 0, False),
            (-1.0, 4, 4, 0, 0, False),
            (1e-2, 6, -1, 0, 1, True),
            (-1.0, 4, 5, 11, 0, False),
            (-1.0, 4, 5, -10, 0, False),
            (-1.0, 4, -1, 10, 0, False),
            (-1.0, 4, -1, -11, 0, False),
            (-1.0, 4, 7, 2, 0, False),
            (1e-1, 2, 8, None, 0, True),
        ]:
            info = {"error": None} if want_err else None
            left, sv, right = decomp.svd_via_eig_truncated(
                x, cutoff=cutoff, cutoff_mode=mode, max_bond=max_bond,
                absorb=absorb, renorm=renorm, info=info)
            key = f"eig__{mname}__{len(eig_cases)}"
            for nm, v in _gauge_free(left, sv, right).items():
                store[f"{key}__{nm}"] = v
            parts = [a for a in (left, right) if a is not None]
            k = (left.shape[1] if left is not None else
                 right.shape[0] if right is not None else sv.shape[0])
            eig_cases.append({
                "key": key, "mat": mname, "cutoff": cutoff, "cutoff_mode": mode,
                "max_bond": max_bond, "absorb": absorb, "renorm": renorm,
                "n_keep": int(k),
                "error": None if info is None else float(info["error"]),
                "has": [left is not None, sv is not None, right is not None]})
    meta["eig_cases"] = eig_cases
    eigh_cases = []
    for mname in ("sym", "psd", "herm"):
        x = mats[mname]
        for kw in [dict(absorb=None), dict(absorb=None, max_bond=6),
                   dict(absorb=-1, cutoff=1e-2, cutoff_mode=4),
                   dict(absorb=1, cutoff=0.2, cutoff_mode=2),
                   dict(absorb=0, positive=1, max_bond=5) if mname == "psd" else dict(absorb=1, max_bond=5),
                   dict(absorb=None, shift=True, cutoff=1e-3, cutoff_mode=3, renorm=2)]:
            left, sv, right = decomp.eigh_truncated(x, **kw)
            key = f"eigh__{mname}__{len(eigh_cases)}"
            for nm, v in _gauge_free(left, sv, right).items():
                store[f"{key}__{nm}"] = v
            eigh_cases.append({"key": key, "mat": mname, "kw": kw,
                               "n_keep": int(left.shape[1])})
    meta["eigh_cases"] = eigh_cases
    rand_cases = []
    for mname, max_bond, absorb in [("lowrank", 4, 0), ("lowrank", 6, 1), ("lowrank", 5, -1),
                                    ("decay", 8, 0), ("decay", 6, None), ("decay", 12, 1),
                                    ("tall", 4, -1), ("wide", 5, 0), ("cplx", 6, 0),
                                    ("decay", 5, 10), ("decay", 5, -11), ("tall", 10, 1)]:
        x = mats[mname]
        left, sv, right = decomp.svd_rand_truncated(x, max_bond=max_bond, absorb=absorb, seed=5)
        sfull = np.linalg.svd(x, compute_uv=False)
        k = (left.shape[1] if left is not None else right.shape[0])
        rec_err = None
        if left is not None and right is not None:
            rec = left @ (np.diag(sv) @ right if sv is not None else right)
            rec_err = float(np.linalg.norm(x - rec))
        rand_cases.append({"mat": mname, "max_bond": max_bond, "absorb": absorb,
                           "n_keep": int(k), "rec_err": rec_err,
                           "optimal_err": float(np.sqrt(np.sum(sfull[k:] ** 2))),
                           "has": [left is not None, sv is not None, right is not None]})
    meta["rand_cases"] = rand_cases
    meta["parse_split_opts"] = []
    for kw in [dict(method="svd:eig"), dict(method="svd:eig", absorb="rfactor", max_bond=5, cutoff=None),
               dict(method="svd:rand", max_bond=7), dict(method="svd:rand", max_bond=7, absorb="left", cutoff=1e-3),
               dict(method="eigh", renorm=True, cutoff_mode="sum1"), dict(method="eigh", absorb=None),
               dict(method="lq"), dict(method="qr", absorb="lorthog")]:
        method, opts = decomp.parse_split_opts(**kw)
        meta["parse_split_opts"].append({"kw": kw, "method": method, "opts": opts})
    meta["svals"] = {}
    for mname in ("tall", "wide", "cplx"):
        store[f"svals__{mname}__svd"] = np.asarray(decomp.array_svals(mats[mname], method="svd"))
        store[f"svals__{mname}__eig"] = np.asarray(decomp.array_svals(mats[mname], method="svd:eig"))
    np.savez_compressed(os.path.join(OUT, "decomp2.npz"), **store)
    json.dump(meta, open(os.path.join(OUT, "decomp2.json"), "w"), indent=1, default=str)


def decomp3_cases():
    """'cholesky', 'qr:cholesky' / 'lq:cholesky' and 'polar_right' / 'polar_left'
    of the reference on its numpy backend (factors are unique: stored as is)."""
    import warnings
    rng = np.random.default_rng(23)
    store, meta = {}, {}
    ps = rng.standard_normal((16, 24))
    hc = rng.standard_normal((12, 18)) + 1j * rng.standard_normal((12, 18))
    big = rng.standard_normal((72, 90))
    mats = {
        "pd": ps @ ps.T / 24,
        "hpd": hc @ hc.conj().T / 18,
        "pd_big": big @ big.T / 90,
        "tall": rng.standard_normal((24, 10)),
        "wide": rng.standard_normal((9, 20)),
        "square": rng.standard_normal((16, 16)),
        "cplx": rng.standard_normal((12, 14)) + 1j * rng.standard_normal((12, 14)),
        "ctall": rng.standard_normal((15, 7)) + 1j * rng.standard_normal((15, 7)),
        "tall_big": rng.standard_normal((150, 70)),
    }
    for k, v in mats.items():
        store[f"mat__{k}"] = v

    def put(key, left, sv, right):
        assert sv is None
        if left is not None:
            store[f"{key}__left"] = np.asarray(left)
        if right is not None:
            store[f"{key}__right"] = np.asarray(right)
        return [left is not None, False, right is not None]

    chol = []
    for mname in ("pd", "hpd", "pd_big"):
        for absorb in (0, -12, 12):
            for shift in (True, False, "auto", 1e-3):
                if mname == "pd_big" and (absorb, shift) not in ((-12, True), (12, False)):
                    continue
                key = f"chol__{len(chol)}"
                has = put(key, *decomp.cholesky_regularized(mats[mname], absorb=absorb, shift=shift))
                chol.append({"key": key, "mat": mname, "absorb": absorb, "shift": shift, "has": has})
    meta["cholesky_cases"] = chol
    qrc = []
    for mname, absorbs in [("tall", (1, 10, 11)), ("wide", (-1, -10, -11)),
                           ("square", (1, 10, 11, -1, -10, -11)), ("cplx", (-1, -10, -11)),
                           ("ctall", (1, 10, 11)), ("tall_big", (11,))]:
        for absorb in absorbs:
            for st in (True, False):
                if mname == "tall_big" and not st:
                    continue
                key = f"qrc__{len(qrc)}"
                has = put(key, *decomp.qr_via_cholesky(mats[mname], absorb=absorb,
                                                       solve_triangular=st))
                qrc.append({"key": key, "mat": mname, "absorb": absorb,
                            "solve_triangular": st, "has": has})
    meta["qr_cholesky_cases"] = qrc
    pol = []
    for mname in ("tall", "wide", "square", "cplx", "ctall"):
        for side in ("right", "left"):
            if (side == "right") != (mats[mname].shape[0] >= mats[mname].shape[1]) and \
                    mats[mname].shape[0] != mats[mname].shape[1]:
                continue    # P would be rank deficient and U not unique
            key = f"polar__{len(pol)}"
            fn = decomp.polar_right if side == "right" else decomp.polar_left
            has = put(key, *fn(mats[mname]))
            pol.append({"key": key, "mat": mname, "side": side, "has": has})
    meta["polar_cases"] = pol
    meta["parse_split_opts"] = []
    for kw in [dict(method="cholesky"), dict(method="cholesky", absorb="lsqrt"),
               dict(method="qr:cholesky"), dict(method="lq:cholesky"),
               dict(method="qr:cholesky", absorb="rfactor"),
               dict(method="polar_right"), dict(method="polar_left", max_bond=4)]:
        method, opts = decomp.parse_split_opts(**kw)
        meta["parse_split_opts"].append({"kw": kw, "method": method, "opts": opts})
    # array_split end to end + error behaviour
    arr = []
    for mname, kw in [("pd", dict(method="cholesky")), ("tall", dict(method="qr:cholesky")),
                      ("wide", dict(method="lq:cholesky")), ("square", dict(method="polar_right")),
                      ("square", dict(method="polar_left"))]:
        key = f"asplit__{len(arr)}"
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            has = put(key, *decomp.array_split(mats[mname], cutoff=0.0, **kw))
        arr.append({"key": key, "mat": mname, "kw": kw, "has": has})
    meta["array_split_cases"] = arr
    errs = {}
    indef = mats["square"] + mats["square"].T
    store["mat__indef"] = indef
    for shift in (False, True, "auto"):
        try:
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                decomp.cholesky_regularized(indef, shift=shift)
            errs[str(shift)] = None
        except Exception as e:  # noqa: BLE001
            errs[str(shift)] = type(e).__name__
    try:
        decomp.parse_split_opts(method="polar_right", absorb=None)
        errs["polar_absorb_none"] = None
    except Exception as e:  # noqa: BLE001
        errs["polar_absorb_none"] = type(e).__name__
    try:
        decomp.cholesky_regularized(mats["pd"], absorb=1)
        errs["chol_bad_absorb"] = None
    except Exception as e:  # noqa: BLE001
        errs["chol_bad_absorb"] = type(e).__name__
    meta["errors"] = errs
    # 'lu' split: (P L, None, U) with weak rows / columns dropped
    lu = []
    lowrank = mats["tall"] @ rng.standard_normal((10, 12))            # 24 x 12, full column rank
    store["mat__lu_mixed"] = np.concatenate([lowrank, 1e-9 * rng.standard_normal((24, 3))], axis=1)
    for mname, kw in [("square", dict()), ("tall", dict(cutoff=1e-12, cutoff_mode=2)),
                      ("wide", dict(cutoff=1e-3, cutoff_mode=1)), ("cplx", dict(cutoff=1e-10, cutoff_mode=2)),
                      ("lu_mixed", dict(cutoff=1e-6, cutoff_mode=2)),
                      ("lu_mixed", dict(cutoff=1e-6, cutoff_mode=1))]:
        key = f"lu__{len(lu)}"
        x = store[f"mat__{mname}"]
        kw2 = dict(cutoff_mode=2, **kw) if "cutoff_mode" not in kw else kw
        has = put(key, *decomp.lu_truncated(x, **kw2))
        lu.append({"key": key, "mat": mname, "kw": kw2, "has": has})
    meta["lu_cases"] = lu
    # diagonal helpers
    d = np.abs(rng.standard_normal(16)) + 0.1
    d[3] = 0.0
    z = rng.standard_normal(9) + 1j * rng.standard_normal(9)
    z[2] = 0.0
    store["helpers__d"] = d
    store["helpers__z"] = z
    store["helpers__rddiv"] = decomp.rddiv(mats["square"], d)
    store["helpers__lddiv"] = decomp.lddiv(d, mats["square"])
    store["helpers__sgn"] = decomp.sgn(z)
    store["helpers__sgn_real"] = decomp.sgn(z.real)
    store["helpers__safe_inverse"] = decomp.safe_inverse(d)
    store["helpers__safe_inverse_sqrt"] = decomp.safe_inverse(d, cutoff=1e-3, power=0.5)
    np.savez_compressed(os.path.join(OUT, "decomp3.npz"), **store)
    json.dump(meta, open(os.path.join(OUT, "decomp3.json"), "w"), indent=1, default=str)


def _dump_tn2d(tn, key, store):
    """Store every tensor of a 2D network: data, index names, site, layer."""
    recs = []
    for k, t in enumerate(tn.tensors):
        site = [tg for tg in t.tags if tg.startswith("I")]
        assert len(site) == 1
        i, j = map(int, site[0][1:].split(","))
        layer = "KET" if "KET" in t.tags else ("BRA" if "BRA" in t.tags else None)
        store[f"{key}__t{k}"] = np.asarray(t.data)
        recs.append({"inds": list(map(str, t.inds)), "site": [i, j], "layer": layer})
    return recs


def boundary_cases():
    """contract_boundary (mode='mps') of the reference on small PEPS norm
    networks (two-layer) and flat 2D networks."""
    store, meta = {}, {}
    nets = {}
    p = qtn.PEPS.rand(4, 4, bond_dim=3, phys_dim=2, seed=4, dtype="complex128")
    nets["peps44"] = (p.make_norm(), ("KET", "BRA"))
    p2 = qtn.PEPS.rand(3, 5, bond_dim=2, phys_dim=2, seed=7, dtype="float64")
    nets["peps35"] = (p2.make_norm(), ("KET", "BRA"))
    p3 = qtn.PEPS.rand(5, 3, bond_dim=2, phys_dim=2, seed=9, dtype="complex64")
    nets["peps53_c64"] = (p3.make_norm(), ("KET", "BRA"))
    nets["flat55"] = (qtn.TN2D_rand(5, 5, D=3, seed=2), None)
    nets["flat64"] = (qtn.TN2D_rand(6, 4, D=2, seed=3, dtype="complex128"), None)
    for name, (tn, layers) in nets.items():
        recs = _dump_tn2d(tn, name, store)
        exact = complex(tn.contract(all, optimize="auto-hq"))
        runs = []
        for kw in [dict(max_bond=4, cutoff=0.0), dict(max_bond=8, cutoff=0.0),
                   dict(max_bond=16, cutoff=0.0), dict(max_bond=8),
                   dict(max_bond=6, cutoff=0.0, sequence=["xmin"]),
                   dict(max_bond=6, cutoff=0.0, sequence=["ymin", "ymax"]),
                   dict(max_bond=5, cutoff=1e-3, sequence=["xmax"]),
                   dict(max_bond=6, cutoff=0.0, canonize=False)]:
            v = complex(tn.contract_boundary(layer_tags=layers, **kw))
            runs.append({"kw": kw, "value": [v.real, v.imag]})
        meta[name] = {"Lx": tn.Lx, "Ly": tn.Ly, "layers": layers, "tensors": recs,
                      "exact": [exact.real, exact.imag], "runs": runs,
                      "dtype": str(tn.dtype)}
    # PEPS site-array convention (for peps_norm_tensors): arrays in site order
    for i in range(4):
        for j in range(4):
            t = p[i, j]
            store[f"peps44_site__{i}_{j}"] = np.asarray(t.data)
    meta["peps44_site_inds"] = {f"{i},{j}": list(map(str, p[i, j].inds))
                                for i in range(4) for j in range(4)}
    meta["peps44_bonds"] = {
        f"{i},{j}": {"up": (str(list(qtn.bonds(p[i, j], p[i + 1, j]))[0]) if i < 3 else None),
                     "right": (str(list(qtn.bonds(p[i, j], p[i, j + 1]))[0]) if j < 3 else None)}
        for i in range(4) for j in range(4)}
    np.savez_compressed(os.path.join(OUT, "boundary.npz"), **store)
    json.dump(meta, open(os.path.join(OUT, "boundary.json"), "w"), indent=1)


def compressed_cases():
    """_contract_compressed_tid_sequence of the reference (compress_mode
    'basic', tree_gauge_distance=0: no tree gauging) on small networks along a
    fixed sequence: final values for several option sets."""
    store, meta = {}, {}
    nets = {
        "flat44": qtn.TN2D_rand(4, 4, D=3, seed=5),
        "flat53_c": qtn.TN2D_rand(5, 3, D=2, seed=6, dtype="complex128"),
        "norm33": qtn.PEPS.rand(3, 3, bond_dim=2, phys_dim=2, seed=8).make_norm(),
        "reg10": qtn.TN_rand_reg(10, 3, D=3, seed=11),
    }
    for name, tn in nets.items():
        tids = list(tn.tensor_map)
        arrays = [np.asarray(tn.tensor_map[t].data) for t in tids]
        inputs = [list(map(str, tn.tensor_map[t].inds)) for t in tids]
        output = list(map(str, tn.outer_inds()))
        # a greedy pairwise sequence (smallest result first): (tid1, tid2) steps,
        # the result lives on under the second id
        sizes = {}
        for a, t in zip(arrays, inputs):
            for ix, d in zip(t, a.shape):
                sizes[ix] = d
        live = {k: set(t) for k, t in enumerate(inputs)}
        seq = []
        while len(live) > 1:
            best = None
            keys = list(live)
            for x in range(len(keys)):
                for y in range(x + 1, len(keys)):
                    a, b = keys[x], keys[y]
                    if not (live[a] & live[b]):
                        continue
                    other = set(output)
                    for k2, v in live.items():
                        if k2 not in (a, b):
                            other |= v
                    res = {ix for ix in (live[a] | live[b]) if ix in other}
                    cost = int(np.prod([sizes[ix] for ix in res])) if res else 1
                    if best is None or cost < best[0]:
                        best = (cost, a, b, res)
            if best is None:          # disconnected: outer product of the first two
                a, b = keys[0], keys[1]
                best = (0, a, b, live[a] | live[b])
            _, a, b, res = best
            seq.append((a, b))
            del live[a]
            del live[b]
            live[b] = res
        exact = tn.contract(all, optimize="auto-hq", output_inds=tn.outer_inds())
        exact = np.asarray(exact.data if hasattr(exact, "data") else exact)
        for k, a in enumerate(arrays):
            store[f"{name}__t{k}"] = a
        runs = []
        for kw in [dict(max_bond=4, cutoff=0.0), dict(max_bond=8, cutoff=0.0),
                   dict(max_bond=6, cutoff=1e-6), dict(max_bond=5, cutoff=0.0, compress_late=False),
                   dict(max_bond=6, cutoff=0.0, compress_span=2),
                   dict(max_bond=6, cutoff=0.0, compress_matrices=False),
                   dict(max_bond=4, cutoff=0.0, equalize_norms=True),
                   dict(max_bond=7, cutoff=0.0, compress_min_size=64)]:
            tn2 = tn.copy()
            res = tn2._contract_compressed_tid_sequence(
                [(tids[a], tids[b]) for a, b in seq], output_inds=tn.outer_inds(),
                tree_gauge_distance=0, compress_mode="basic", **kw)
            val = np.asarray(res.data if hasattr(res, "data") else res)
            if hasattr(res, "inds"):
                val = np.asarray(res.transpose(*tn.outer_inds()).data)
            key = f"{name}__run{len(runs)}"
            store[key] = val
            runs.append({"kw": kw, "key": key})
        store[f"{name}__exact"] = exact
        meta[name] = {"inputs": inputs, "output": output, "seq": [list(s) for s in seq],
                      "runs": runs, "dtype": str(tn.dtype)}
    np.savez_compressed(os.path.join(OUT, "compressed.npz"), **store)
    json.dump(meta, open(os.path.join(OUT, "compressed.json"), "w"), indent=1)


def tebd_cases():
    """gate_split / gate_with_auto_swap / TEBD of the reference (numpy)."""
    store, meta = {}, {}
    rng = np.random.default_rng(21)
    # --- gate_split on a random MPS --------------------------------------
    p = qtn.MPS_rand_state(6, 5, seed=8, dtype="complex128")
    for i in range(6):
        store[f"gs_mps__{i}"] = np.asarray(p[i].data)
    meta["gs_mps_inds"] = [list(map(str, p[i].inds)) for i in range(6)]
    G = rng.standard_normal((4, 4)) + 1j * rng.standard_normal((4, 4))
    store["gs_gate"] = G
    gs = []
    for kw in [dict(where=(2, 3)), dict(where=(2, 3), max_bond=3, cutoff=0.0, absorb="right"),
               dict(where=(3, 2), absorb="left"), dict(where=(0, 1), cutoff=1e-2, cutoff_mode="rel"),
               dict(where=(4, 5), max_bond=2)]:
        q = p.copy()
        q.canonicalize_(kw["where"])
        q.gate_split_(G, **kw)
        key = f"gs__{len(gs)}"
        store[key + "__dense"] = np.asarray(q.to_dense()).reshape(-1)
        gs.append({"key": key, "kw": {k: (list(v) if k == "where" else v) for k, v in kw.items()},
                   "bond": int(q.bond_size(*sorted(kw["where"])))})
    meta["gate_split"] = gs
    sw = []
    for where in [(1, 4), (4, 1), (0, 5), (2, 3)]:
        q = p.copy()
        q.gate_with_auto_swap_(G, where, cutoff=1e-12)
        key = f"swap__{len(sw)}"
        store[key + "__dense"] = np.asarray(q.to_dense()).reshape(-1)
        sw.append({"key": key, "where": list(where)})
    meta["auto_swap"] = sw
    # --- TEBD -------------------------------------------------------------
    runs = []
    for L, order, dt, T, imag, bz in [(8, 4, 0.05, 0.4, False, 0.0), (7, 2, 0.02, 0.1, False, 0.3),
                                      (8, 2, 0.1, 1.0, True, 0.0), (6, 4, None, 0.3, False, 0.0)]:
        H = qtn.ham_1d_heis(L, bz=bz, cyclic=False)
        p0 = qtn.MPS_neel_state(L)
        kw = dict(dt=dt) if dt is not None else dict(tol=1e-3)
        tebd = qtn.TEBD(p0, H, progbar=False, imag=imag,
                        split_opts=dict(cutoff=1e-12), **kw)
        tebd.update_to(T, order=order)
        pt = tebd.pt
        key = f"tebd__{len(runs)}"
        store[key + "__dense"] = np.asarray(pt.to_dense()).reshape(-1)
        terms = {f"{a},{b}": np.asarray(h) for (a, b), h in H.terms.items()}
        for k2, h in terms.items():
            store[f"{key}__term__{k2}"] = h
        runs.append({"key": key, "L": L, "order": order, "dt": dt, "T": T, "imag": imag,
                     "bz": bz, "tol": None if dt is not None else 1e-3,
                     "terms": sorted(terms), "err": float(tebd.err), "t": float(tebd.t),
                     "max_bond": int(pt.max_bond()),
                     "energy": float(np.real(qtn.expec_TN_1D(pt.H, qtn.MPO_ham_heis(L, bz=bz), pt)
                                             / (pt.H @ pt)))})
    meta["tebd"] = runs
    store["heis_h2"] = np.asarray(qu.ham_heis(2, cyclic=False))
    meta["trotter"] = {str(o): [[int(k), float(f)] for k, f in
                                __import__("quimb.tensor.tnag.tebd", fromlist=["x"]).trotter_schedule(2, o)]
                       for o in (1, 2, 4)}
    np.savez_compressed(os.path.join(OUT, "tebd.npz"), **store)
    json.dump(meta, open(os.path.join(OUT, "tebd.json"), "w"), indent=1)


def mps_ops_cases():
    """MPS compression / addition / MPO application / overlap of the reference."""
    store, meta = {}, {}
    p = qtn.MPS_rand_state(7, 6, seed=31, dtype="complex128")
    q = qtn.MPS_rand_state(7, 3, seed=32, dtype="float64")
    H = qtn.MPO_ham_heis(7)
    for i in range(7):
        store[f"p__{i}"] = np.asarray(p[i].data)
        store[f"q__{i}"] = np.asarray(q[i].data)
        store[f"H__{i}"] = np.asarray(H[i].data)
    meta["p_inds"] = [list(map(str, p[i].inds)) for i in range(7)]
    meta["H_inds"] = [list(map(str, H[i].inds)) for i in range(7)]
    meta["overlap_pq"] = [float(np.real(p.H @ q)), float(np.imag(p.H @ q))]
    store["p_dense"] = np.asarray(p.to_dense()).reshape(-1)
    store["add_dense"] = np.asarray((p + q).to_dense()).reshape(-1)
    Hp = H.apply(p)
    store["Hp_dense"] = np.asarray(Hp.to_dense()).reshape(-1)
    meta["Hp_bonds"] = [int(Hp.bond_size(i, i + 1)) for i in range(6)]
    cases = []
    for kw in [dict(form="right", max_bond=3, cutoff=0.0), dict(form="left", max_bond=3, cutoff=0.0),
               dict(form=2, max_bond=4, cutoff=0.0), dict(form=5, cutoff=1e-2),
               dict(form="flat", max_bond=3, cutoff=0.0), dict(cutoff=1e-1, cutoff_mode="rel"),
               dict(form="left", max_bond=2, cutoff=0.0, method="svd:eig")]:
        c = Hp.copy()
        c.compress(**kw)
        key = f"cmp__{len(cases)}"
        store[key + "__dense"] = np.asarray(c.to_dense()).reshape(-1)
        cases.append({"key": key, "kw": kw,
                      "bonds": [int(c.bond_size(i, i + 1)) for i in range(6)]})
    meta["compress"] = cases
    np.savez_compressed(os.path.join(OUT, "mps_ops.npz"), **store)
    json.dump(meta, open(os.path.join(OUT, "mps_ops.json"), "w"), indent=1)


def mps_dmrg_cases():
    store, meta = {}, {}
    # Heisenberg MPO of the reference, as arrays (lrud layout) + dense check
    H = qtn.MPO_ham_heis(6)
    for i in range(6):
        store[f"heis6__{i}"] = np.asarray(H[i].data)
    meta["heis6_inds"] = [list(map(str, H[i].inds)) for i in range(6)]
    store["heis6__dense"] = np.asarray(H.to_dense())
    # MPS norm / expectation
    p = qtn.MPS_rand_state(12, 7, seed=3, normalize=False)
    for i in range(12):
        store[f"mps12__{i}"] = np.asarray(p[i].data)
    meta["mps12_inds"] = [list(map(str, p[i].inds)) for i in range(12)]
    meta["mps12_norm2"] = float(p.H @ p)
    meta["mps12_norm"] = float(p.norm())
    H12 = qtn.MPO_ham_heis(12)
    meta["mps12_expec_heis"] = float(qtn.expec_TN_1D(p.H, H12, p))
    # complex MPS
    pc = qtn.MPS_rand_state(8, 5, seed=4, normalize=False, dtype="complex128")
    for i in range(8):
        store[f"cmps8__{i}"] = np.asarray(pc[i].data)
    meta["cmps8_norm2"] = float(np.real(pc.H @ pc))
    meta["cmps8_expec_heis"] = float(np.real(qtn.expec_TN_1D(pc.H, qtn.MPO_ham_heis(8), pc)))
    # DMRG2 energies of the reference itself
    runs = []
    for L, bond_dims, cutoffs, tol in [(10, [8, 16, 32], 1e-10, 1e-8),
                                       (20, [10, 20, 40], 1e-10, 1e-6),
                                       (32, [16, 32], 1e-9, 1e-6)]:
        Hm = qtn.MPO_ham_heis(L)
        dm = qtn.DMRG2(Hm, bond_dims=bond_dims, cutoffs=cutoffs)
        conv = dm.solve(tol=tol, max_sweeps=8, verbosity=0)
        exact = None
        if L <= 14:
            exact = float(qu.groundenergy(qu.ham_heis(L, cyclic=False, sparse=True)))
        runs.append({"L": L, "bond_dims": bond_dims, "cutoffs": cutoffs, "tol": tol,
                     "converged": bool(conv), "energies": [float(e) for e in dm.energies],
                     "exact": exact, "max_bond": int(dm.state.max_bond())})
    meta["dmrg2_runs"] = runs
    # DMRG1 of the reference (bond expansion noise is unseeded there: energies
    # are compared at the convergence tolerance, not bit-wise)
    runs1 = []
    for L, bond_dims, tol in [(10, [4, 8, 16, 32], 1e-8), (16, [8, 16, 32], 1e-7)]:
        Hm = qtn.MPO_ham_heis(L)
        dm1 = qtn.DMRG1(Hm, bond_dims=bond_dims, cutoffs=1e-10)
        conv = dm1.solve(tol=tol, max_sweeps=12, verbosity=0)
        exact = float(qu.groundenergy(qu.ham_heis(L, cyclic=False, sparse=True)))
        runs1.append({"L": L, "bond_dims": bond_dims, "tol": tol, "converged": bool(conv),
                      "energies": [float(e) for e in dm1.energies], "exact": exact,
                      "max_bond": int(dm1.state.max_bond())})
    meta["dmrg1_runs"] = runs1
    meta["heisenberg_energy_100_periodic"] = float(qu.heisenberg_energy(100))
    np.savez_compressed(os.path.join(OUT, "mps_dmrg.npz"), **store)
    json.dump(meta, open(os.path.join(OUT, "mps_dmrg.json"), "w"), indent=1)


DROPIN_SPLITS = [
    ("svd", dict(cutoff=1e-3, cutoff_mode="rel")), ("svd", dict(max_bond=3, absorb="left")),
    ("svd:eig", dict(max_bond=4)), ("qr", {}), ("lq", {}), ("eigh", dict(max_bond=4)),
    ("polar_right", {}), ("polar_left", {}),
]


def dropin_cases():
    """What the drop-in tests compare the backend with: the names the
    reference's composed drivers accept registrations for, and its own numpy
    runs of Tensor @ / tensor_contract / Tensor.split and of the drivers
    either side of the hot path, with the inputs they ran on."""
    import warnings
    from quimb.linalg import base_linalg
    from quimb.tensor import array_ops
    store, meta = {}, {}
    meta["registrable"] = {
        "decomp": sorted(nm for nm, f in vars(decomp).items() if hasattr(f, "register")),
        "array_ops": sorted(nm for nm, f in vars(array_ops).items() if hasattr(f, "register")),
        "split_values": sorted(decomp._SPLIT_VALUES_FNS),
        "eigs_methods": sorted(base_linalg._EIGS_METHODS),
    }
    rng = np.random.default_rng(0)
    shapes = {"a": ((4, 5, 6), "abc"), "b": ((6, 5, 7), "cbd"), "c": ((7, 3), "de"),
              "h1": ((3, 4), "xh"), "h2": ((4, 5), "hy"), "h3": ((4, 2), "hz")}
    ts = {}
    for k, (shape, inds) in shapes.items():
        store[f"contract__{k}"] = rng.standard_normal(shape)
        ts[k] = qtn.Tensor(store[f"contract__{k}"], inds=inds)
    for k, (shape, inds) in {"z1": ((3, 4), "ab"), "z2": ((4, 3), "ba")}.items():
        store[f"contract__{k}"] = rng.standard_normal(shape) + 1j * rng.standard_normal(shape)
        ts[k] = qtn.Tensor(store[f"contract__{k}"], inds=inds)
    meta["contract_inds"] = {k: list(t.inds) for k, t in ts.items()}
    ab = ts["a"] @ ts["b"]
    store["contract__ab"] = np.asarray(ab.data)
    meta["contract_ab_inds"] = list(ab.inds)
    store["contract__abc_ea"] = np.asarray(
        qtn.tensor_contract(ts["a"], ts["b"], ts["c"], output_inds="ea").data)
    store["contract__hyper_xyz"] = np.asarray(
        qtn.tensor_contract(ts["h1"], ts["h2"], ts["h3"], output_inds="xyz").data)
    z = complex(qtn.tensor_contract(ts["z1"], ts["z2"]))
    m, e = qtn.tensor_contract(ts["z1"], ts["z2"], strip_exponent=True)
    meta["contract_z"] = [z.real, z.imag]
    meta["contract_z_strip"] = {"mantissa": [complex(m).real, complex(m).imag],
                                "exponent": float(e)}
    splits = []
    for k, (method, kw) in enumerate(DROPIN_SPLITS):
        rng = np.random.default_rng(1)
        x = rng.standard_normal((6, 4, 5))
        if method == "eigh":
            y = rng.standard_normal((6, 4, 6, 4))
            x = y + y.transpose(2, 3, 0, 1)
            inds, left = "abcd", ["a", "b"]
        else:
            inds = "abc"
            left = ["a", "b"] if method in ("qr", "polar_right") else ["a"]
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ref = qtn.Tensor(x, inds=inds).split(left_inds=left, method=method,
                                                 get="arrays", **kw)
        store[f"split{k}__x"] = x
        store[f"split{k}__product"] = np.tensordot(ref[0], ref[-1], 1)
        splits.append({"method": method, "kw": kw, "inds": inds, "left_inds": left,
                       "shapes": [list(r.shape) for r in ref]})
    meta["splits"] = splits
    _dropin_callers(store, meta)
    np.savez_compressed(os.path.join(OUT, "dropin.npz"), **store)
    json.dump(meta, open(os.path.join(OUT, "dropin.json"), "w"), indent=1)


def _store_tn(tn, key, store):
    """Every tensor of a network: data under key__t<k>, index names returned."""
    inds = []
    for k, t in enumerate(tn.tensors):
        store[f"{key}__t{k}"] = np.asarray(t.data)
        inds.append(list(map(str, t.inds)))
    return inds


def _dropin_callers(store, meta):
    """The reference's drivers either side of the hot path, on numpy: MPS
    canonize / compress / expectation, TNLinearOperator, DMRG2 (both local
    eigensolver forms), boundary contraction, circuit amplitude, TEBD, DMRG1,
    MPS gates / MPO application / addition / entropy, compressed contraction."""
    import warnings
    from quimb.tensor.tensor_core import TNLinearOperator
    warnings.simplefilter("ignore")

    def sites(p, key):
        for i in range(p.L):
            store[f"{key}__{i}"] = np.asarray(p[i].data)       # 'lrp', ends (r,p)/(l,p)

    def mpo(H, key):
        for i in range(H.L):
            store[f"{key}__{i}"] = np.asarray(H[i].data)       # 'lrud'

    # canonize / compress / expectation / linear operator
    p = qtn.MPS_rand_state(6, 7, seed=4)
    sites(p, "canon_p")
    c = {"norm0": float(p.H @ p)}
    p.left_canonize()
    c["norm_canon"] = float(p.H @ p)
    p.compress(max_bond=3)
    c["norm_compressed"] = float(p.H @ p)
    c["max_bond"] = int(p.max_bond())
    H = qtn.MPO_ham_heis(6)
    mpo(H, "heis6")
    c["expec"] = float(qtn.expec_TN_1D(p.H, H, p))
    rng = np.random.default_rng(2)
    ts = [qtn.Tensor(rng.standard_normal((5, 3, 5)), inds=("a", "w", "b"), tags="L"),
          qtn.Tensor(rng.standard_normal((3, 2, 2)), inds=("w", "p", "q"), tags="W")]
    A = TNLinearOperator(ts, left_inds=("a", "p"), right_inds=("b", "q"))
    v = rng.standard_normal(10)
    for k, t in enumerate(ts):
        store[f"linop__t{k}"] = np.asarray(t.data)
    store["linop__v"] = v
    store["linop__matvec"] = A.matvec(v)
    store["linop__dense"] = A.to_dense()
    meta["canon"] = c

    # DMRG2, L = 8: quimb's default eigensolver path and both dense settings
    L = 8
    H8 = qtn.MPO_ham_heis(L)
    mpo(H8, "heis8")
    p4 = qtn.MPS_rand_state(L, 4, seed=3)
    p8 = qtn.MPS_rand_state(L, 8, seed=3)
    sites(p4, "dmrg_p4")
    sites(p8, "dmrg_p8")
    d = {}
    ref = qtn.DMRG2(H8.copy(), bond_dims=[8, 16, 32], cutoffs=1e-10, p0=p4.copy())
    ref.solve(tol=1e-8, max_sweeps=5, verbosity=0)
    d["default_energy"] = float(ref.energy)
    for dense in (True, False):
        ref = qtn.DMRG2(H8.copy(), bond_dims=[8, 16], cutoffs=1e-10, p0=p8.copy())
        ref.opts["local_eig_ham_dense"] = dense
        ref.solve(tol=1e-9, max_sweeps=5, verbosity=0)
        d[f"dense_{dense}"] = {"energy": float(ref.energy),
                               "bonds": [int(ref.state.bond_size(i, i + 1)) for i in range(L - 1)]}
    d["exact"] = float(qu.groundenergy(qu.ham_heis(L, cyclic=False, sparse=True)))
    r1 = qtn.DMRG1(H8.copy(), bond_dims=[8, 16], p0=p8.copy())
    r1.solve(tol=1e-8, max_sweeps=4, verbosity=0)
    d["dmrg1_energy"] = float(r1.energy)
    meta["dmrg"] = d

    cl = {}
    # PEPS norm by boundary-MPS contraction; classical Ising partition function
    peps = qtn.PEPS.rand(4, 4, bond_dim=2, seed=1, dtype="complex128")
    for i in range(4):
        for j in range(4):
            store[f"peps__{i}_{j}"] = np.asarray(peps[i, j].data)
    v = complex(peps.make_norm().contract_boundary(max_bond=8, cutoff=0.0,
                                                   layer_tags=("KET", "BRA")))
    cl["peps_norm"] = [v.real, v.imag]
    ising = qtn.TN2D_classical_ising_partition_function(4, 4, beta=0.3)
    cl["ising_tensors"] = _dump_tn2d(ising, "ising", store)
    cl["ising_Z"] = float(ising.contract_boundary(max_bond=8))

    # circuit amplitude
    rng = np.random.default_rng(0)
    circ = qtn.Circuit(5)
    for dd in range(4):
        for q in range(5):
            circ.apply_gate("U3", *rng.uniform(0, 6, 3), q)
        for q in range(dd % 2, 4, 2):
            circ.apply_gate("CZ", q, q + 1)
    amp = complex(circ.amplitude("01001"))
    cl["amp_01001"] = [amp.real, amp.imag]
    # the networks unsimplified: quimb's default simplification reduces these
    # to the amplitude itself, which would leave nothing to contract
    cl["amp_01001_inds"] = _store_tn(circ.amplitude_tn("01001", simplify_sequence=""),
                                     "amp_01001", store)
    tn = circ.amplitude_tn("00000", simplify_sequence="")
    cl["amp_00000_inds"] = _store_tn(tn, "amp_00000", store)
    amp = complex(tn.full_simplify() ^ all)
    cl["amp_00000"] = [amp.real, amp.imag]

    # TEBD from the Neel state
    ham = qtn.ham_1d_heis(6)
    store["tebd__h2"] = np.asarray(ham.terms[(0, 1)])
    cl["tebd_terms_equal"] = all(np.allclose(ham.terms[k], ham.terms[(0, 1)]) for k in ham.terms)
    t0 = qtn.TEBD(qtn.MPS_neel_state(6), ham, progbar=False)
    t0.update_to(0.2, dt=0.05, order=2)
    store["tebd__dense"] = np.asarray(t0.pt.to_dense()).reshape(-1)

    # MPS gates, MPO application, addition, entropy
    p = qtn.MPS_rand_state(6, 4, seed=2)
    q = qtn.MPS_rand_state(6, 3, seed=6)
    sites(p, "gates_p")
    sites(q, "gates_q")
    G = qu.rand_uni(4, seed=1).reshape(2, 2, 2, 2)
    store["gates__G"] = np.asarray(G)
    for where, fn in (((2, 3), "gate_split"), ((0, 4), "gate_with_auto_swap")):
        store[f"gates__{fn}"] = np.asarray(getattr(p, fn)(G, where, cutoff=1e-12).to_dense()).reshape(-1)
    store["gates__apply"] = np.asarray(H.apply(p).to_dense()).reshape(-1)
    store["gates__add"] = np.asarray((p + q).to_dense()).reshape(-1)
    cl["entropy3"] = float(p.entropy(3))
    meta["callers"] = cl

    # compressed contraction along an inward sequence; max_bond below D, so
    # that every run truncates (the value differs from the exact contraction)
    tn = qtn.TN2D_rand(4, 4, D=4, seed=5)
    tids = list(tn.tensor_map)
    for k, t in enumerate(tids):
        store[f"compressed__t{k}"] = np.asarray(tn.tensor_map[t].data)
    seq_pos = [(i, i + 1) for i in range(len(tids) - 1)]
    seq = [(tids[a], tids[b]) for a, b in seq_pos]
    runs = []
    for kw in (dict(max_bond=3, cutoff=0.0, tree_gauge_distance=0, compress_mode="basic"),
               dict(max_bond=3, cutoff=1e-8, tree_gauge_distance=0, compress_mode="basic",
                    compress_late=False)):
        val = tn.copy()._contract_compressed_tid_sequence(seq, output_inds=(), **kw)
        runs.append({"kw": kw, "value": float(val)})
    meta["compressed"] = {"inputs": [list(map(str, tn.tensor_map[t].inds)) for t in tids],
                          "seq": seq_pos, "runs": runs, "exact": float(tn.contract(all))}


if __name__ == "__main__":
    only = set(sys.argv[1:])
    for fn in (contract_cases, decomp_cases, decomp2_cases, decomp3_cases, boundary_cases, compressed_cases,
               tebd_cases, mps_ops_cases, mps_dmrg_cases, dropin_cases):
        if not only or fn.__name__ in only:
            fn()
    print("golden fixtures written to", OUT)
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))
