"""CPU: the oracle (oracle/cp_oracle.py + cd_oracle.c) against (a) golden vectors produced by the
reference's own code (oracle/make_golden.py) and (b) scikit-learn itself."""
import os

import numpy as np
import pytest

import cases
import cp_oracle as O


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name), allow_pickle=False)


@pytest.mark.parametrize("name", list(cases.DICTIONARY_CASES))
@pytest.mark.parametrize("form", ["dense", "gram"])
def test_dictionary_matches_reference_golden(golden_dir, name, form):
    spec = cases.DICTIONARY_CASES[name]
    g = _load(golden_dir, "dictionary_%s.npz" % name)
    X, W2, Y = cases.case_inputs(spec)
    np.testing.assert_array_equal(g["checksum"], [X.sum(dtype=np.float64), W2.sum(dtype=np.float64), Y.sum()])
    st = O.DictState(alpha=spec["alpha0"], rank_tol=spec.get("rank_tol", .1))
    np.random.seed(spec["np_seed"])
    idxs, W, B = O.dictionary(X.astype(np.float64), W2, Y, rank=spec["rank"], B2=np.zeros(W2.shape[0]), state=st,
                              form=form)
    after = np.random.randint(0, 1 << 30)
    assert np.array_equal(idxs, g["idxs"])  # selected-channel set: exact
    assert after == int(g["rng_after"])  # same number of global RNG draws as the reference
    assert st.alpha == float(g["alpha_final"])
    assert W.shape == g["W"].shape
    # same LAPACK driver as the reference -> identical up to threading order
    assert np.linalg.norm(W - g["W"]) <= 1e-9 * np.linalg.norm(g["W"])
    assert np.abs(B - g["B"]).max() <= 1e-9 * max(1.0, np.abs(g["B"]).max())


def test_golden_versions_recorded(golden_dir):
    """The goldens and the coordinate-descent control flow are those of the third-party versions recorded next to
    them; a different installed scikit-learn is reported (the sklearn cross-checks below may then differ, the goldens
    stay authoritative)."""
    import json

    import sklearn
    v = json.load(open(os.path.join(golden_dir, "VERSIONS.json")))
    assert set(v) == {"scikit-learn", "scipy", "numpy"}
    if sklearn.__version__ != v["scikit-learn"]:
        pytest.skip("installed scikit-learn %s differs from the goldens' %s" % (sklearn.__version__, v["scikit-learn"]))


def test_lasso_cd_matches_sklearn():
    from sklearn.linear_model import Lasso

    X, W2, Y = cases.dictionary_inputs(c=48, n=24, N=800, k=3, seed=3)
    N, c = X.shape[0], X.shape[1]
    samples = np.random.RandomState(0).randint(0, N, 40)
    reX = np.rollaxis(X.reshape((N, c, -1))[samples], 1, 0).astype(np.float64)
    reW2 = np.transpose(W2.reshape((24, c, -1)), [1, 2, 0])
    Z = np.matmul(reX, reW2).reshape((c, -1)).T
    y = Y[samples].reshape(-1)
    sk = Lasso(alpha=1e-3, warm_start=True, selection='random')
    for form in ("dense", "gram"):
        mine = O.LassoCD(alpha=1e-3, form=form)
        sk = Lasso(alpha=1e-3, warm_start=True, selection='random')
        for a in (1e-3, 4e-3, 1.6e-2, 8e-3):
            np.random.seed(17)
            sk.alpha = a
            sk.fit(Z, y)
            np.random.seed(17)
            mine.alpha = a
            mine.fit(Z, y)
            assert mine.n_iter_ == sk.n_iter_
            assert np.array_equal(mine.coef_ != 0, sk.coef_ != 0)
            np.testing.assert_allclose(mine.coef_, sk.coef_, rtol=0, atol=1e-11 * np.abs(sk.coef_).max())
            assert abs(mine.intercept_ - sk.intercept_) < 1e-10


def test_rand_r_sequence():
    import ctypes

    lib = O._clib()
    s = ctypes.c_uint32(12345)
    got = [lib.cp_our_rand_r(ctypes.byref(s)) for _ in range(5)]

    def ref(seed):
        out = []
        for _ in range(5):
            seed ^= (seed << 13) & 0xFFFFFFFF
            seed ^= seed >> 17
            seed ^= (seed << 5) & 0xFFFFFFFF
            out.append(seed % (2147483647 + 1))
        return out

    assert got == ref(12345)


def test_linear_regression_matches_sklearn():
    from sklearn.linear_model import LinearRegression

    r = np.random.RandomState(2)
    for (N, K, n) in [(300, 40, 7), (50, 90, 5)]:  # over- and under-determined
        X = r.standard_normal((N, K))
        Y = r.standard_normal((N, n))
        reg = LinearRegression().fit(X, Y)
        coef, b = O.fc_kernel(X, Y)
        np.testing.assert_allclose(coef, reg.coef_, atol=1e-10)
        np.testing.assert_allclose(b, reg.intercept_, atol=1e-10)


def _forward_from(images, specs, weights, biases):
    from make_golden import conv2d_numpy

    cache = {}

    def forward(batch):
        if batch not in cache:
            blobs = {"data": images[batch % len(images)]}
            for s in specs:
                y = conv2d_numpy(blobs[s["bottom"]], weights[s["name"]], biases[s["name"]], s["pad"], s["stride"])
                blobs[s["name"]] = y
                blobs[s["name"] + "_relu"] = np.maximum(y, 0)
            cache[batch] = blobs
        return cache[batch]

    return forward


@pytest.mark.parametrize("name", list(cases.NET_CASES))
def test_gathers_match_reference_golden(golden_dir, name):
    spec = cases.NET_CASES[name]
    g = _load(golden_dir, "net_%s.npz" % name)
    images, specs, weights, biases = cases.net_inputs(**spec["gen"])
    forward = _forward_from(images, specs, weights, biases)
    names = [s["name"] for s in specs]
    np.random.seed(spec["np_seed"])
    feats, points = O.extract_features(forward, names, spec["nBatches"], spec["P"])
    for nm in names:
        assert feats[nm].dtype == np.float64
        np.testing.assert_array_equal(feats[nm], g["feats_" + nm])  # bit exact
        for b in range(spec["nBatches"]):
            np.testing.assert_array_equal(points[(b, nm, "randx")], g["randx_%s_%d" % (nm, b)])
            np.testing.assert_array_equal(points[(b, nm, "randy")], g["randy_%s_%d" % (nm, b)])
    s2 = specs[1]
    yspec = O.ConvSpec(s2["name"], s2["bottom"], s2["k"], s2["pad"], s2["stride"])
    XY = O.extract_XY(forward, spec["xy"][0], yspec, points)
    np.testing.assert_array_equal(XY, g["XY"])  # bit exact
    if spec.get("dictionary_kernel"):
        st = O.DictState(alpha=1e-3)
        np.random.seed(spec["np_seed"] + 1)
        idxs, W, B = O.dictionary_kernel(forward, spec["xy"][0], yspec, weights["conv2"], biases["conv2"],
                                         feats["conv2"], points, int(g["dk_dprime"]), state=st)
        assert np.array_equal(idxs, g["dk_idxs"])
        assert st.alpha == float(g["dk_alpha"])
        assert np.linalg.norm(W - g["dk_W"]) <= 1e-9 * np.linalg.norm(g["dk_W"])
        assert np.abs(B - g["dk_B"]).max() <= 1e-9


def test_patch_invariant():
    """The reference's own debug check (lib/net.py:659-679): relu(patch) . W2 + b2 == conv output."""
    spec = cases.NET_CASES["k3s2"]
    images, specs, weights, biases = cases.net_inputs(**spec["gen"])
    forward = _forward_from(images, specs, weights, biases)
    np.random.seed(1)
    feats, points = O.extract_features(forward, ["conv2"], spec["nBatches"], spec["P"])
    s2 = specs[1]
    XY = O.extract_XY(forward, "conv1", O.ConvSpec("conv2", "conv1_relu", s2["k"], s2["pad"], s2["stride"]), points)
    k = s2["k"]
    X = np.rollaxis(XY.reshape((-1, k, k, XY.shape[1])), 3, 1)
    fake = O.relu(X).reshape(X.shape[0], -1) @ weights["conv2"].reshape(weights["conv2"].shape[0], -1).T + biases["conv2"]
    assert np.abs(fake - feats["conv2"]).max() < 1e-4  # CHECK_EQ tolerance, lib/utils.py:75-82


# ---------------------------------------------------------------------------- 3C companions (VH / ITQ)
def _sign_align(a, b, axis):
    """Singular vectors are defined up to sign: flips slices of ``a`` along ``axis`` to agree with ``b``."""
    a2 = np.moveaxis(a, axis, 0).copy()
    b2 = np.moveaxis(b, axis, 0)
    for k in range(a2.shape[0]):
        if np.vdot(a2[k], b2[k]) < 0:
            a2[k] = -a2[k]
    return np.moveaxis(a2, 0, axis)


@pytest.mark.parametrize("name", list(cases.VH_CASES))
def test_vh_decompose_matches_reference_golden(golden_dir, name):
    spec = cases.VH_CASES[name]
    g = np.load(os.path.join(golden_dir, "%s.npz" % name))
    W, X, Y = cases.vh_inputs(**spec["gen"])
    V, H, VHr, b = O.VH_decompose(W.astype(np.float64), rank=spec["rank"], X=X.astype(np.float64), Y=Y)
    assert V.shape == g["V"].shape and H.shape == g["H"].shape and VHr.shape == g["VHr"].shape
    np.testing.assert_allclose(VHr, g["VHr"], rtol=0, atol=1e-9 * np.abs(g["VHr"]).max())
    np.testing.assert_allclose(b, g["b"], rtol=0, atol=1e-9)
    np.testing.assert_allclose(_sign_align(V, g["V"], 0), g["V"], rtol=0, atol=1e-9)
    np.testing.assert_allclose(_sign_align(H, g["H"], 1), g["H"], rtol=0, atol=1e-8 * np.abs(g["H"]).max())
    V0, H0, VHr0 = O.VH_decompose(W.astype(np.float64), rank=spec["rank"])
    np.testing.assert_allclose(VHr0, g["VHr0"], rtol=0, atol=1e-12)


@pytest.mark.parametrize("name", list(cases.ITQ_CASES))
def test_itq_decompose_matches_reference_golden(golden_dir, name):
    spec = cases.ITQ_CASES[name]
    g = np.load(os.path.join(golden_dir, "%s.npz" % name))
    feat, gt, H, VHr, bias = cases.itq_inputs(**spec["gen"])
    W1, W2, B, W12 = O.ITQ_decompose(feat, gt, H, spec["rank"], bias=bias, Wr=VHr)
    assert W1.shape == g["W1"].shape and W2.shape == g["W2"].shape
    np.testing.assert_allclose(W12, g["W12"], rtol=0, atol=1e-8 * np.abs(g["W12"]).max())
    np.testing.assert_allclose(B, g["B"], rtol=0, atol=1e-8)
    np.testing.assert_allclose(_sign_align(W1, g["W1"], 0), g["W1"], rtol=0, atol=1e-7 * np.abs(g["W1"]).max())
    np.testing.assert_allclose(_sign_align(W2, g["W2"], 1), g["W2"], rtol=0, atol=1e-7 * np.abs(g["W2"]).max())


class StageSync:
    """R3 checkpoint hook (cp_oracle.R3 / cpb200 Net.R3): at every point where the reference enters one of its three
    per-layer solvers -- and at the end -- compares the live parameters with the snapshot the reference run left in the
    golden (oracle/make_golden.py: run_r3_cases) and, when ``put`` is given, replaces them with the reference's
    (teacher forcing: every stage then starts from the reference's exact state, so its own deviation is measured
    instead of the compounded one)."""

    def __init__(self, golden, get, put, tol):
        self.g, self.get, self.put, self.tol = golden, get, put, tol
        self.i, self.worst, self.log = 0, 0.0, []

    def __call__(self, stage):
        stages = [str(x) for x in self.g["snap_stages"]]
        assert self.i < len(stages) and stage == stages[self.i], (self.i, stage, stages)
        pre = "snap__%d__" % self.i
        for key in [k for k in self.g if k.startswith(pre)]:
            kind, nm = key[len(pre):].split("__")
            ref = self.g[key]
            live = np.asarray(self.get(kind, nm), dtype=np.float64)
            if kind == "w":
                e = float(np.linalg.norm(live - ref) / max(np.linalg.norm(ref), 1e-30))
            else:
                e = float(np.abs(live - ref).max() / max(1.0, np.abs(ref).max()))
            self.log.append((self.i, stage, kind, nm, e))
            self.worst = max(self.worst, e)
            assert e <= self.tol, (self.i, stage, kind, nm, e)
            if self.put is not None:
                self.put(kind, nm, ref)
        self.i += 1

    def done(self):
        return self.i == len(self.g["snap_stages"])


def r3_compare(golden, WPQ, selection, weights, biases, tol_inv=1e-6, tol_fac=1e-5):
    """Compares an R3 outcome with the reference's golden: selections exactly; sign-invariant quantities (live
    weights/biases, the P-layer biases) tightly; the individual V / H / P factors up to the sign of each component."""
    for k in [k for k in golden if k.startswith("sel__")]:
        assert np.array_equal(selection[k[5:]], golden[k]), k
    worst = 0.0
    for k in [k for k in golden if k.startswith("w__")]:
        nm = k[3:]
        e = np.linalg.norm(weights[nm] - golden[k]) / np.linalg.norm(golden[k])
        eb = np.abs(biases[nm] - golden["b__" + nm]).max() / max(1.0, np.abs(golden["b__" + nm]).max())
        worst = max(worst, e, eb)
        assert e <= tol_inv and eb <= tol_inv, (nm, e, eb)
    for k in [k for k in golden if k.startswith("WPQ__")]:
        parts = k[5:].split("__")
        key = (parts[0], int(parts[1])) if len(parts) == 2 else parts[0]
        got, ref = np.asarray(WPQ[key]), golden[k]
        assert got.shape == ref.shape, (key, got.shape, ref.shape)
        if isinstance(key, tuple) and key[1] == 1:     # biases: sign invariant (H bias is zeros, P bias = B)
            assert np.abs(got - ref).max() <= tol_inv * max(1.0, np.abs(ref).max()), key
            continue
        name = key if isinstance(key, str) else key[0]
        # V: (rank, c, h, 1) components along axis 0; H after ITQ = W1 (d', r, 1, w) components along axis 0 AND axis 1;
        # P = W2 (n', d', 1, 1) components along axis 1: compare through sign-insensitive Gram matrices
        a, b = got.reshape(got.shape[0], -1), ref.reshape(ref.shape[0], -1)
        if name.endswith("_V"):
            inv_a, inv_b = a.T @ a, b.T @ b            # projector onto the kept spatial components
        elif name.endswith("_P"):
            inv_a, inv_b = a @ a.T, b @ b.T
        else:
            inv_a, inv_b = np.abs(a), np.abs(b)        # |entries| are invariant to both sign families
        assert np.linalg.norm(inv_a - inv_b) <= tol_fac * np.linalg.norm(inv_b), key
    return worst


@pytest.mark.parametrize("name", list(cases.R3_CASES))
def test_r3_walk_matches_reference_golden(golden_dir, name):
    spec = cases.R3_CASES[name]
    g = cases.load_r3_golden(golden_dir, name)
    images, specs, weights, biases = cases.r3_inputs(**spec["gen"])
    net = O.NumpyNet(specs, weights, biases)
    np.random.seed(spec["np_seed"])
    # freeze: sample points + features once (net.py:749-800), images kept under (batch, 0)
    pd0 = {}
    fwd = lambda b: net.forward_blobs(images[b % len(images)])  # noqa: E731
    feats, pd = O.extract_features(fwd, net.convs, spec["nBatches"], spec["P"])
    for b in range(spec["nBatches"]):
        pd[(b, 0)] = images[b % len(images)]
    for nm in net.convs:
        assert cases.digest(feats[nm]) == g["sha256__feats__" + nm], nm
    net._feats_dict, net._points_dict = feats, pd
    st = O.DictState(alpha=1e-3)
    sync = StageSync(g, lambda kind, nm: (net.weights if kind == "w" else net.biases)[nm], None, tol=1e-6)
    WPQ = O.R3(net, state=st, checkpoint=sync)
    assert sync.done()
    assert st.alpha == float(g["alpha_final"])
    assert np.random.randint(0, 1 << 30) == int(g["rng_after"])
    r3_compare(g, WPQ, net.selection, net.weights, net.biases)
