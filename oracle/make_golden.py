"""TEST INFRASTRUCTURE: generates tests/golden/*.npz by running the UNMODIFIED reference
(/root/reference/lib/decompose.py and lib/net.py, imported through oracle/ref_shims.py) on
small seeded inputs.  Runs only in the build container (the reference is Python and cannot
travel to the GPU box); the fixtures it writes are committed.

    python oracle/make_golden.py            # rewrites tests/golden/

What is pinned
  dictionary_*.npz   outputs of reference ``dictionary`` (mask, weights, bias, final cfgs.alpha)
                     for inputs regenerated from a seed by tests/cases.py
  net_*.npz          outputs of reference ``Net.extract_features`` / ``Net.extract_XY`` /
                     ``Net.dictionary_kernel`` driven through a duck-typed Net (no Caffe): a tiny
                     two-conv network whose forward pass is computed with numpy.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import ref_shims  # noqa: E402
import cases  # noqa: E402  (tests/cases.py)

OUT = os.path.join(ROOT, "tests", "golden")


def run_dictionary_cases(D, CF):
    for name, spec in cases.DICTIONARY_CASES.items():
        X, W2, Y = cases.case_inputs(spec)
        CF.alpha = spec["alpha0"]
        CF.c.dic.rank_tol = spec.get("rank_tol", .1)
        np.random.seed(spec["np_seed"])
        idxs, W, B = D.dictionary(X.astype(np.float64), W2, Y, rank=spec["rank"], B2=np.zeros(W2.shape[0]))
        after = np.random.randint(0, 1 << 30)  # pins how many global draws the reference consumed
        np.savez_compressed(os.path.join(OUT, "dictionary_%s.npz" % name), idxs=idxs, W=W, B=B,
                            alpha_final=CF.alpha, rng_after=after,
                            checksum=np.array([X.sum(dtype=np.float64), W2.sum(dtype=np.float64), Y.sum()]))
        Xs = X[:, idxs].reshape(X.shape[0], -1).astype(np.float64)
        sv = np.linalg.svd(Xs - Xs.mean(0), compute_uv=False)
        print(name, "kept", int(idxs.sum()), "of", len(idxs), "alpha", CF.alpha,
              "cond(centred Gram of kept columns) %.2e" % ((sv[0] / sv[-1]) ** 2))
    CF.c.dic.rank_tol = .1


def conv2d_numpy(x, w, b, pad, stride):
    """fp32 direct convolution (what Caffe's forward would give up to rounding)."""
    B, c, H, W = x.shape
    n, _, k, _ = w.shape
    xp = np.zeros((B, c, H + 2 * pad, W + 2 * pad), dtype=np.float32)
    xp[:, :, pad:H + pad, pad:W + pad] = x
    Ho, Wo = (H + 2 * pad - k) // stride + 1, (W + 2 * pad - k) // stride + 1
    out = np.zeros((B, n, Ho, Wo), dtype=np.float32)
    for i in range(Ho):
        for j in range(Wo):
            patch = xp[:, :, i * stride:i * stride + k, j * stride:j * stride + k].reshape(B, -1)
            out[:, :, i, j] = patch @ w.reshape(n, -1).T + b
    return out


def make_fake_net(NET, CF, images, specs, weights, biases):
    """A reference ``Net`` whose Caffe accessors are replaced by numpy state."""

    class _Inner:  # stands in for pycaffe's net object
        def __init__(self, outer):
            self.outer = outer

        def set_input_arrays(self, data, label):
            self.outer._cur = (data, label)

    class FakeNet(NET.Net):
        def __init__(self):
            self._mem = True
            self.net = _Inner(self)
            self._batch_iter = 0
            self._cur = None
            self._blobs = {}
            self.convs = [s["name"] for s in specs if s.get("type") != "pool"]
            self.innerproduct, self.sums, self.bns = [], [], []
            self._bottom_names = {s["name"]: [s["bottom"]] for s in specs}  # backs the bottom_names property
            self.num = images[0].shape[0]
            self.acc = []
            self.forward()  # dry pass: Caffe knows blob shapes statically
            self._shapes = {k: v.shape for k, v in self._blobs.items()}
            self._batch_iter = 0

        def forward(self):
            if self._cur is None:  # first (non-frozen) pass draws the next batch itself
                data = images[self._batch_iter % len(images)]
                label = np.zeros((data.shape[0], 1, 1, 1), dtype=np.float32)
                self._batch_iter += 1
            else:
                data, label = self._cur
            self._data, self._label = data, label
            blobs = {"data": data}
            for s in specs:
                if s.get("type") == "pool":  # 2x2 / stride 2 max pooling (VGG)
                    x = blobs[s["bottom"]]
                    Bq, cq, Hq, Wq = x.shape
                    blobs[s["name"]] = x[:, :, :Hq // 2 * 2, :Wq // 2 * 2].reshape(Bq, cq, Hq // 2, 2, Wq // 2, 2).max((3, 5))
                    continue
                y = conv2d_numpy(blobs[s["bottom"]], weights[s["name"]], biases[s["name"]], s["pad"], s["stride"])
                blobs[s["name"]] = y
                blobs[s["name"] + "_relu"] = np.maximum(y, 0)
            self._blobs = blobs
            self._cur = None
            return {}

        def data(self):
            return self._data

        def label(self):
            return self._label

        def clr_acc(self):
            pass

        def blobs_data(self, name): return self._blobs[name]
        def blobs_shape(self, name): return self._shape(name)
        def blobs_num(self, name): return self._shape(name)[0]
        def blobs_channels(self, name): return self._shape(name)[1]
        def blobs_height(self, name): return self._shape(name)[2]
        def blobs_width(self, name): return self._shape(name)[3]
        def blobs_type(self, name): return np.float32

        def _shape(self, name):
            return self._shapes[name]

        def _sp(self, name): return [s for s in specs if s["name"] == name][0]
        def conv_param_pad(self, name): return self._sp(name)["pad"]
        def conv_param_kernel_size(self, name): return self._sp(name)["k"]
        def conv_param_stride(self, name): return self._sp(name)["stride"]
        def param_shape(self, name): return weights[name].shape
        def param_data(self, name): return weights[name]
        def param_b_data(self, name): return biases[name]
        def set_param_data(self, name, data): weights[name][...] = data.copy()   # net.py:213-217
        def set_param_b(self, name, data): biases[name][...] = data.copy()       # net.py:219-220
        def appresb(self, name): return 0  # dcfgs.res.short == 0 (net.py:1648)
        # prototxt surgery of R3 (net.py:884-966, 321-366, 161-164): no numerical effect, nothing to edit here
        def insert(self, *a, **k): pass
        def set_conv(self, *a, **k): pass
        def infer_pad_kernel(self, W, origin_name): return {}
        def save_pt(self, *a, **k): return "pt"

    return FakeNet()


def run_net_cases(NET, CF, D):
    for name, spec in cases.NET_CASES.items():
        images, specs, weights, biases = cases.net_inputs(**spec["gen"])
        CF.c.nBatches = spec["nBatches"]
        CF.c.nPointsPerLayer = spec["P"]
        CF.c.dic.option = 0
        CF.c.dic.fitfc = 0
        CF.c.model = ''
        CF.alpha = 1e-3
        net = make_fake_net(NET, CF, images, specs, weights, biases)
        np.random.seed(spec["np_seed"])
        names = [s["name"] for s in specs]
        feats_dict, points_dict = net.extract_features(names, save=1)
        net.load_frozen(feats_dict=feats_dict, points_dict=points_dict)
        x_name, y_name = spec["xy"]
        XY = net.extract_XY(x_name, y_name)
        out = dict(XY=XY)
        for nm in names:
            out["feats_" + nm] = feats_dict[nm]
            for b in range(spec["nBatches"]):
                out["randx_%s_%d" % (nm, b)] = points_dict[(b, nm, "randx")]
                out["randy_%s_%d" % (nm, b)] = points_dict[(b, nm, "randy")]
        if spec.get("dictionary_kernel"):
            c_out = weights[x_name].shape[0]
            d_prime = int(c_out / 1.15)
            np.random.seed(spec["np_seed"] + 1)
            idxs, W2n, B2n = net.dictionary_kernel(x_name, None, d_prime, y_name, None)
            out.update(dk_idxs=idxs, dk_W=W2n, dk_B=B2n, dk_alpha=CF.alpha, dk_dprime=d_prime)
            print(name, "dictionary_kernel kept", int(idxs.sum()), "of", len(idxs))
        np.savez_compressed(os.path.join(OUT, "net_%s.npz" % name), **out)
        print(name, "XY", XY.shape, {k: v.shape for k, v in feats_dict.items()})


def run_r3_cases(NET, CF, D):
    """The reference's own Net.R3 (VH -> ITQ -> channel pruning per layer, sequential, error compensating) on a tiny
    VGG-named stack.  Outputs: every WPQ entry, the selections, the final weights / biases of the live net."""
    for name, spec in cases.R3_CASES.items():
        images, specs, weights, biases = cases.r3_inputs(**spec["gen"])
        CF.c.nBatches = spec["nBatches"]
        CF.c.nPointsPerLayer = spec["P"]
        CF.c.dic.option = 0
        CF.c.dic.fitfc = 0
        CF.c.dic.vh = 1
        CF.c.dic.keep = 3.
        CF.c.model = ''
        CF.alpha = 1e-3
        net = make_fake_net(NET, CF, images, specs, weights, biases)
        np.random.seed(spec["np_seed"])
        feats_dict, points_dict = net.extract_features(net.convs, save=1)
        net.load_frozen(feats_dict=feats_dict, points_dict=points_dict)
        # Stage snapshots: the live weights / biases on ENTRY of each of the three per-layer solvers (and at the end).
        # The walk is error compensating, so a deviation in one stage feeds the next through features of nearly
        # rank-deficient blobs; the snapshots let a test re-synchronise an implementation stage by stage
        # (tests/test_gpu_r3.py: teacher-forced walk) instead of comparing only the compounded end result.
        snaps = []

        def snap(stage):
            snaps.append((stage, {nm: weights[nm].copy() for nm in net.convs}, {nm: biases[nm].copy() for nm in net.convs}))

        def wrap(fn, stage):
            def inner(*a, **k):
                snap(stage)
                return fn(*a, **k)
            return inner

        orig_vh, orig_itq = NET.VH_decompose, NET.ITQ_decompose
        NET.VH_decompose, NET.ITQ_decompose = wrap(orig_vh, "vh"), wrap(orig_itq, "itq")
        net.dictionary_kernel = wrap(net.dictionary_kernel, "prune")
        try:
            WPQ, new_pt = net.R3()
        finally:
            NET.VH_decompose, NET.ITQ_decompose = orig_vh, orig_itq
        snap("final")
        out = {"snap_stages": np.array([st for st, _, _ in snaps])}
        prev_w, prev_b = {}, {}
        for i, (st, w_, b_) in enumerate(snaps):  # only what changed since the previous snapshot
            for nm in net.convs:
                if nm not in prev_w or not np.array_equal(prev_w[nm], w_[nm]):
                    out["snap__%d__w__%s" % (i, nm)] = w_[nm]
                if nm not in prev_b or not np.array_equal(prev_b[nm], b_[nm]):
                    out["snap__%d__b__%s" % (i, nm)] = b_[nm]
            prev_w, prev_b = w_, b_
        for k, v in WPQ.items():
            out["WPQ__" + ("%s__%d" % k if isinstance(k, tuple) else k)] = np.asarray(v)
        for k, v in net.selection.items():
            out["sel__" + k] = v
        for nm in net.convs:
            out["w__" + nm] = weights[nm]
            out["b__" + nm] = biases[nm]
            out["feats__" + nm] = feats_dict[nm]
        out["alpha_final"] = CF.alpha
        out["rng_after"] = np.random.randint(0, 1 << 30)
        np.savez_compressed(os.path.join(OUT, "%s.npz" % name), **cases.compact_r3_golden(out, spec))
        print(name, "WPQ keys", sorted(str(k) for k in WPQ), "kept", {k: int(v.sum()) for k, v in net.selection.items()},
              "alpha", CF.alpha)


def run_3c_cases(D, CF):
    """VH_decompose (with its nonlinear_fc refit) and ITQ_decompose of the reference on small seeded inputs."""
    for name, spec in cases.VH_CASES.items():
        W, X, Y = cases.vh_inputs(**spec["gen"])
        V, H, VHr, b = D.VH_decompose(W.astype(np.float64), rank=spec["rank"], DEBUG=0, X=X.astype(np.float64), Y=Y)
        V0, H0, VHr0 = D.VH_decompose(W.astype(np.float64), rank=spec["rank"])
        np.savez_compressed(os.path.join(OUT, "%s.npz" % name), V=V, H=H, VHr=VHr, b=b, V0=V0, H0=H0, VHr0=VHr0)
        print(name, "V", V.shape, "H", H.shape, "VHr", VHr.shape)
    for name, spec in cases.ITQ_CASES.items():
        feat, gt, H, VHr, bias = cases.itq_inputs(**spec["gen"])
        W1, W2, B, W12 = D.ITQ_decompose(feat, gt, H, spec["rank"], bias=bias, DEBUG=0, Wr=VHr)
        np.savez_compressed(os.path.join(OUT, "%s.npz" % name), W1=W1, W2=W2, B=B, W12=W12)
        print(name, "W1", W1.shape, "W2", W2.shape, "W12", W12.shape)


def write_versions():
    """The reference pins no versions of its third-party solvers (README.md:46); the goldens -- and the control flow the
    LASSO kernel reproduces bit for bit (gap-safe screening, stopping rule) -- are those of the versions recorded here."""
    import json

    import scipy
    import sklearn
    with open(os.path.join(OUT, "VERSIONS.json"), "w") as f:
        json.dump({"scikit-learn": sklearn.__version__, "scipy": scipy.__version__, "numpy": np.__version__}, f, indent=1)


def main():
    os.makedirs(OUT, exist_ok=True)
    D, NET, CF = ref_shims.load_reference()
    assert NET is not None, ref_shims._loaded.get("net_error")
    run_dictionary_cases(D, CF)
    run_net_cases(NET, CF, D)
    run_3c_cases(D, CF)
    run_r3_cases(NET, CF, D)
    write_versions()


if __name__ == "__main__":
    main()
