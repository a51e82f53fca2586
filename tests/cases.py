"""Seeded input generators shared by oracle/make_golden.py (which runs the real reference on
them) and the tests (which regenerate the same inputs and compare against the stored
reference outputs).  numpy's legacy RandomState stream is stable across versions."""
import hashlib
import os

import numpy as np


def dictionary_inputs(c, n, N, k, seed, noise=0.01):
    """X (N,c,k,k) fp32 post-ReLU patches, W2 (n,c,k,k) fp32, Y (N,n) float64 holding fp32 values."""
    r = np.random.RandomState(seed)
    X = np.maximum(r.standard_normal((N, c, k, k)).astype(np.float32), 0)
    W2 = (r.standard_normal((n, c, k, k)) * np.sqrt(2.0 / (c * k * k))).astype(np.float32)
    Y = X.reshape(N, -1).astype(np.float64) @ W2.reshape(n, -1).T.astype(np.float64)
    Y = Y + noise * Y.std() * r.standard_normal(Y.shape)
    Y = Y.astype(np.float32).astype(np.float64)
    return X, W2, Y


def correlated_inputs(c, n, N, k, seed, noise=0.01, H=20, collinear=None):
    """Realistic conditioning: post-ReLU features of a random 3x3 conv over SMOOTH images (low-pass filtered
    noise), so that channels and neighbouring taps are strongly correlated (cond of the centred Gram >= 1e4,
    against ~1e1-1e3 for the iid inputs above).  ``collinear=(a, b, eps)`` makes channel b an almost exact
    multiple of channel a (relative perturbation eps).  Same return convention as dictionary_inputs."""
    r = np.random.RandomState(seed)
    nimg = -(-N // 16)
    img = r.standard_normal((nimg, 3, H + 8, H + 8))
    for _ in range(3):  # separable box blur, three passes ~ gaussian
        img = (img + np.roll(img, 1, 2) + np.roll(img, -1, 2)) / 3.0
        img = (img + np.roll(img, 1, 3) + np.roll(img, -1, 3)) / 3.0
    img = (img / img.std()).astype(np.float32)
    w1 = (r.standard_normal((c, 3, 3, 3)) * np.sqrt(2.0 / 27)).astype(np.float32)
    b1 = (0.1 * r.standard_normal(c)).astype(np.float32)
    Hf = H + 6
    feat = np.zeros((nimg, c, Hf, Hf), dtype=np.float32)
    for dy in range(3):
        for dx in range(3):
            feat += np.einsum("bchw,oc->bohw", img[:, :, dy:dy + Hf, dx:dx + Hf], w1[:, :, dy, dx]).astype(np.float32)
    feat = np.maximum(feat + b1[None, :, None, None], 0).astype(np.float32)
    if collinear is not None:
        a, b, eps = collinear
        feat[:, b] = (feat[:, a] * np.float32(1.5) * (1 + eps * r.standard_normal(feat[:, a].shape))).astype(np.float32)
    ys = r.randint(0, Hf - k + 1, N)
    xs = r.randint(0, Hf - k + 1, N)
    ims = r.randint(0, nimg, N)
    X = np.stack([feat[i, :, y:y + k, x:x + k] for i, y, x in zip(ims, ys, xs)]).astype(np.float32)
    W2 = (r.standard_normal((n, c, k, k)) * np.sqrt(2.0 / (c * k * k))).astype(np.float32)
    Y = X.reshape(N, -1).astype(np.float64) @ W2.reshape(n, -1).T.astype(np.float64)
    Y = Y + noise * Y.std() * r.standard_normal(Y.shape)
    Y = Y.astype(np.float32).astype(np.float64)
    return X, W2, Y


def case_inputs(spec):
    """Inputs of a DICTIONARY_CASES entry (iid generator unless the case names another one)."""
    if spec.get("generator") == "correlated":
        return correlated_inputs(**spec["gen"])
    return dictionary_inputs(**spec["gen"])


DICTIONARY_CASES = {
    # name: generator args, target rank, np.random.seed before the call, cfgs.alpha on entry
    "c32": dict(gen=dict(c=32, n=16, N=600, k=3, seed=11), rank=27, np_seed=5, alpha0=1e-3),
    "c64": dict(gen=dict(c=64, n=48, N=1000, k=3, seed=12), rank=55, np_seed=6, alpha0=1e-3),
    "k1": dict(gen=dict(c=96, n=32, N=800, k=1, seed=13), rank=83, np_seed=7, alpha0=1e-3),
    "full": dict(gen=dict(c=3, n=8, N=400, k=3, seed=14), rank=3, np_seed=8, alpha0=1e-3),  # rank == c shortcut
    "under": dict(gen=dict(c=64, n=16, N=400, k=3, seed=15), rank=55, np_seed=9, alpha0=1e-3),  # N-1 < K'
    "carry": dict(gen=dict(c=48, n=24, N=800, k=3, seed=16), rank=41, np_seed=10, alpha0=0.016),  # carried alpha
    "tol2": dict(gen=dict(c=40, n=24, N=800, k=3, seed=17), rank=30, np_seed=11, alpha0=1e-3, rank_tol=.2),
    # rank_tol >= 1 is an ABSOLUTE slack on the channel count (decompose.py:493-494): window [24, 27]
    "tolabs": dict(gen=dict(c=36, n=20, N=700, k=3, seed=18), rank=24, np_seed=12, alpha0=1e-3, rank_tol=3),
    # correlated (real-conv-like) features: ill-conditioned least squares, the regime of real networks
    "corr": dict(generator="correlated", gen=dict(c=32, n=24, N=1600, k=3, seed=19), rank=27, np_seed=13, alpha0=1e-3),
    "corrbig": dict(generator="correlated", gen=dict(c=48, n=32, N=2400, k=3, seed=20), rank=41, np_seed=14,
                    alpha0=1e-3),
    # one channel an almost exact multiple of another (relative perturbation 1e-4): near-collinear columns
    "collin": dict(generator="correlated", gen=dict(c=24, n=16, N=1200, k=3, seed=21, collinear=(3, 11, 1e-4)),
                   rank=20, np_seed=15, alpha0=1e-3, w_tol=5e-5),
}


def net_inputs(B, H, c1, c2, k, pad, stride, nimgbatches, seed):
    """A two-conv network: data (B,3,H,H) -> conv1 (3->c1, 3x3 pad 1) -> ReLU -> conv2 (c1->c2, k, pad, stride)."""
    r = np.random.RandomState(seed)
    images = [r.standard_normal((B, 3, H, H)).astype(np.float32) for _ in range(nimgbatches)]
    specs = [dict(name="conv1", bottom="data", k=3, pad=1, stride=1),
             dict(name="conv2", bottom="conv1_relu", k=k, pad=pad, stride=stride)]
    weights = {"conv1": (r.standard_normal((c1, 3, 3, 3)) * np.sqrt(2.0 / 27)).astype(np.float32),
               "conv2": (r.standard_normal((c2, c1, k, k)) * np.sqrt(2.0 / (c1 * k * k))).astype(np.float32)}
    biases = {"conv1": (0.1 * r.standard_normal(c1)).astype(np.float32),
              "conv2": (0.1 * r.standard_normal(c2)).astype(np.float32)}
    return images, specs, weights, biases


NET_CASES = {
    "k3s1": dict(gen=dict(B=4, H=12, c1=24, c2=12, k=3, pad=1, stride=1, nimgbatches=6, seed=21), nBatches=6, P=10,
                 np_seed=31, xy=("conv1", "conv2"), dictionary_kernel=True),
    "k3s2": dict(gen=dict(B=3, H=11, c1=8, c2=6, k=3, pad=1, stride=2, nimgbatches=3, seed=22), nBatches=3, P=5,
                 np_seed=32, xy=("conv1", "conv2")),
    "k5s1": dict(gen=dict(B=2, H=9, c1=6, c2=5, k=5, pad=2, stride=1, nimgbatches=3, seed=23), nBatches=3, P=4,
                 np_seed=33, xy=("conv1", "conv2")),
    "k1s1": dict(gen=dict(B=3, H=8, c1=10, c2=7, k=1, pad=0, stride=1, nimgbatches=2, seed=24), nBatches=2, P=6,
                 np_seed=34, xy=("conv1", "conv2")),
}


def vh_inputs(c, n, N, k, seed, noise=0.05):
    """Inputs of VH_decompose as Net.R3 calls it (lib/net.py:1355-1362): weights (n,c,k,k) fp32, X (N,c,k,k) patches of
    the layer's bottom blob, Y (N,n) = sampled output features minus bias (pre-ReLU, both signs)."""
    r = np.random.RandomState(seed)
    X = np.maximum(r.standard_normal((N, c, k, k)).astype(np.float32), 0)
    W = (r.standard_normal((n, c, k, k)) * np.sqrt(2.0 / (c * k * k))).astype(np.float32)
    Y = X.reshape(N, -1).astype(np.float64) @ W.reshape(n, -1).T.astype(np.float64)
    Y = (Y + noise * Y.std() * r.standard_normal(Y.shape)).astype(np.float32).astype(np.float64)
    return W, X, Y


VH_CASES = {
    "vh_small": dict(gen=dict(c=12, n=20, N=900, k=3, seed=41), rank=14),
    "vh_wide": dict(gen=dict(c=24, n=16, N=1500, k=3, seed=42), rank=22),
}


def itq_inputs(n, rvh, c, N, seed, k=3):
    """Inputs of ITQ_decompose as Net.R3 calls it (lib/net.py:1387-1389): feature = features of the layer after the
    spatial decomposition (N,n), gt_feature = the frozen original features, weight = H (n, rvh, 1, k), Wr = VHr."""
    r = np.random.RandomState(seed)
    base = r.standard_normal((N, n // 2)) @ r.standard_normal((n // 2, n)) + 0.3 * r.standard_normal((N, n))
    gt = (base + 0.2).astype(np.float32).astype(np.float64)
    feat = (gt + 0.05 * r.standard_normal((N, n))).astype(np.float32).astype(np.float64)
    H = (r.standard_normal((n, rvh, 1, k)) * 0.2).astype(np.float64)
    VHr = (r.standard_normal((n, c, k, k)) * 0.1).astype(np.float64)
    bias = (0.1 * r.standard_normal(n)).astype(np.float32)
    return feat, gt, H, VHr, bias


ITQ_CASES = {
    "itq_small": dict(gen=dict(n=20, rvh=9, c=8, N=700, seed=51), rank=11),
    "itq_mid": dict(gen=dict(n=48, rvh=20, c=16, N=1600, seed=52), rank=30),
}


def r3_inputs(B, H, widths, nimgbatches, seed):
    """A small VGG-named stack for Net.R3 (lib/net.py:1292-1471 hard-codes the VGG-16 layer names in alldic / pooldic
    / rankdic): data (B,3,H,H) -> conv1_1 -> ReLU -> conv1_2 -> ReLU -> pool1 (2x2/2 max) -> conv2_1 -> ReLU -> conv2_2.
    widths = output channels of the four convs."""
    r = np.random.RandomState(seed)
    images = [r.standard_normal((B, 3, H, H)).astype(np.float32) for _ in range(nimgbatches)]
    names = ["conv1_1", "conv1_2", "conv2_1", "conv2_2"]
    bottoms = ["data", "conv1_1_relu", "pool1", "conv2_1_relu"]
    specs = []
    for nm, bt in zip(names, bottoms):
        specs.append(dict(name=nm, bottom=bt, k=3, pad=1, stride=1))
        if nm == "conv1_2":
            specs.append(dict(name="pool1", bottom="conv1_2_relu", type="pool"))
    weights, biases = {}, {}
    cin = 3
    for nm, co in zip(names, widths):
        weights[nm] = (r.standard_normal((co, cin, 3, 3)) * np.sqrt(2.0 / (cin * 9))).astype(np.float32)
        biases[nm] = (0.1 * r.standard_normal(co)).astype(np.float32)
        cin = co
    return images, specs, weights, biases


R3_CASES = {
    # rankdic x 4/3 (keep = 3): conv1_2 22, conv2_1 49, conv2_2 62 -- widths chosen so that rank <= n and that the
    # `if d_c < rank: d_c = rank` floor (net.py:1349) is exercised at conv2_1 (int(56/1.15) = 48 < 49)
    # conv2_2 is kept wide (96, like VGG's 2:1 ratio of width to rank): truncating 64 channels to rank 62 sits on a
    # near-degenerate pair of singular values, where the reference's own result moves with LAPACK's rounding
    "r3_small": dict(gen=dict(B=4, H=12, widths=(12, 28, 56, 96), nimgbatches=20, seed=61), nBatches=20, P=10,
                     np_seed=71),
}


def digest(a):
    """sha256 of an array's shape and values (as float64, -0.0 taken as 0.0): equal digests <=> equal arrays, the
    condition np.testing.assert_array_equal checks."""
    a = np.ascontiguousarray(a, dtype=np.float64) + 0.0
    h = hashlib.sha256(repr(a.shape).encode())
    h.update(a.tobytes())
    return h.hexdigest()


def _r3_first_snapshot(spec):
    """The live weights / biases the R3 walk starts from: the case's seeded inputs."""
    _, _, weights, biases = r3_inputs(**spec["gen"])
    return {"snap__0__%s__%s" % (kind, nm): v[nm] for kind, v in (("w", weights), ("b", biases)) for nm in v}


def _r3_expand(stored, spec):
    g = dict(stored)
    for k, v in _r3_first_snapshot(spec).items():
        assert digest(v) == str(g.pop("sha256__" + k)), "the seeded inputs no longer reproduce the golden's " + k
        g[k] = v
    for i in range(len(g["snap_stages"])):  # the final state of a layer is its latest snapshot
        for k in [k for k in g if k.startswith("snap__%d__" % i)]:
            kind, nm = k.split("__")[2:]
            g["%s__%s" % (kind, nm)] = g[k]
    return g


def compact_r3_golden(full, spec):
    """What the golden file of an R3 case stores of the full record (oracle/make_golden.py: run_r3_cases), to stay small:
    the sampled features and the first snapshot (the seeded inputs) as digests, and no final w__ / b__ (the latest
    snapshot of each layer).  load_r3_golden rebuilds the record; the features stay digests (sha256__feats__<layer>),
    compared with digest()."""
    out = {}
    for k, v in full.items():
        if k.startswith(("feats__", "snap__0__")):
            out["sha256__" + k] = digest(v)
        elif not k.startswith(("w__", "b__")):
            out[k] = v
    back = _r3_expand(out, spec)
    assert all(np.array_equal(back[k], v) for k, v in full.items() if not k.startswith("feats__")), "lossy"
    return out


def load_r3_golden(golden_dir, name):
    """The reference's R3 record of R3_CASES[name] as a dict (see compact_r3_golden)."""
    with np.load(os.path.join(golden_dir, "%s.npz" % name)) as z:
        return _r3_expand({k: z[k] for k in z.files}, R3_CASES[name])
