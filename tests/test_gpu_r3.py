"""GPU: Net.R3 -- the reference's whole 3C walk (spatial decomposition, channel decomposition, channel pruning, each
stage re-extracting features through the weights the previous ones rewrote) -- against the golden written by the
reference's OWN Net.R3 (oracle/make_golden.py: run_r3_cases), plus the frozen-points pickle round trip."""
import pickle

import numpy as np
import pytest

import cases
import cp_oracle as O
from test_oracle import StageSync, r3_compare

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


class NumpyConvForward:
    """Feature provider computing the blobs with the same fp32 numpy convolution the golden run used (so that the
    sampled features are bit-identical to the reference run); weights are read from the live net."""

    def __init__(self, images, specs):
        self.images, self.specs = images, specs

    def data(self, batch):
        return self.images[batch % len(self.images)]

    def __call__(self, net, data, upto=None):
        data = data.cpu().numpy() if isinstance(data, torch.Tensor) else np.asarray(data, dtype=np.float32)
        blobs = {"data": data}
        for s in self.specs:
            if s.get("type") == "pool":
                x = blobs[s["bottom"]]
                B, c, H, W = x.shape
                blobs[s["name"]] = x[:, :, :H // 2 * 2, :W // 2 * 2].reshape(B, c, H // 2, 2, W // 2, 2).max((3, 5))
                continue
            w = net.param_data(s["name"]).cpu().numpy()
            b = net.param_b_data(s["name"]).cpu().numpy()
            y = O.conv2d_numpy(blobs[s["bottom"]], w, b, s["pad"], s["stride"])
            blobs[s["name"]] = y
            blobs[s["name"] + "_relu"] = np.maximum(y, 0)
        return {k: torch.as_tensor(v, device=net.eng.device) for k, v in blobs.items()}


def build_net(engine, spec, provider_cls, frozen=None):
    from cpb200.lib import net as cpnet

    images, specs, weights, biases = cases.r3_inputs(**spec["gen"])
    convspecs = [s for s in specs if s.get("type") != "pool"]
    cs = [cpnet.ConvSpec(s["name"], s["bottom"], weights[s["name"]].shape[0], s["k"], s["pad"], s["stride"],
                         pool_after=(s["name"] == "conv1_2")) for s in convspecs]
    if provider_cls is NumpyConvForward:
        provider = NumpyConvForward(images, specs)
    else:
        provider = cpnet.ConvStackForward(lambda b: torch.as_tensor(images[b % len(images)], device=engine.device))
    return cpnet.Net(cs, weights, biases, provider, pool_names={"conv1_2": "pool1"}, frozen=frozen), images


def _frozen_net(engine, golden_dir, name, mode):
    from cpb200.lib import cfgs

    spec = cases.R3_CASES[name]
    g = cases.load_r3_golden(golden_dir, name)
    engine.gram_mode = mode
    net, images = build_net(engine, spec, NumpyConvForward)
    cfgs.c.nBatches, cfgs.c.nPointsPerLayer = spec["nBatches"], spec["P"]
    cfgs.c.dic.vh, cfgs.c.dic.keep = 1, 3.
    cfgs.alpha = 1e-3
    np.random.seed(spec["np_seed"])
    feats_dict, points_dict = net.freeze()
    for nm in net.convs:
        assert cases.digest(feats_dict[nm]) == g["sha256__feats__" + nm], nm  # same points, same features
    assert points_dict["data"] == tuple(images[0].shape) and (0, 0) in points_dict and (0, 1) in points_dict
    return spec, g, net, images


@pytest.mark.parametrize("mode", [0, 1], ids=["fp64", "3xtf32"])
@pytest.mark.parametrize("name", list(cases.R3_CASES))
def test_r3_stage_by_stage_against_reference_golden(engine, golden_dir, name, mode):
    """Every stage of the walk (spatial decomposition, channel decomposition, channel pruning -- per layer) started from
    the reference's own live state at that point: weights within 1e-4 relative Frobenius, biases within 1e-4, the
    selections, the alpha carried between layers and the RNG consumption exactly, the V / H / P factors up to sign."""
    from cpb200.lib import cfgs

    spec, g, net, images = _frozen_net(engine, golden_dir, name, mode)
    dev = engine.device

    def get(kind, nm):
        return (net._w if kind == "w" else net._b)[nm].cpu().numpy()

    def put(kind, nm, ref):
        (net._w if kind == "w" else net._b)[nm].copy_(torch.as_tensor(ref, device=dev))

    sync = net._checkpoint = StageSync(g, get, put, tol=1e-4)
    WPQ, new_pt = net.R3()
    assert sync.done()
    assert cfgs.alpha == float(g["alpha_final"])
    assert np.random.randint(0, 1 << 30) == int(g["rng_after"])  # the walk consumed the reference's RNG draws
    weights = {k: v.cpu().numpy() for k, v in net._w.items()}
    biases = {k: v.cpu().numpy() for k, v in net._b.items()}
    r3_compare(g, WPQ, net.selection, weights, biases, tol_inv=1e-4, tol_fac=1e-4)
    assert new_pt["prefix"] == "3C4x" and [l["V"] for l in new_pt["layers"]] == ["conv1_2_V", "conv2_1_V", "conv2_2_V"]
    print("R3 %s mode %d, stage by stage: worst deviation %.2e\n  " % (name, mode, sync.worst) +
          "\n  ".join("%d %-5s %s %-8s %.2e" % e for e in sync.log))


@pytest.mark.parametrize("mode", [0, 1], ids=["fp64", "3xtf32"])
@pytest.mark.parametrize("name", list(cases.R3_CASES))
def test_r3_free_running_walk(engine, golden_dir, name, mode):
    """The same walk left alone.  The blobs behind an approximated layer are nearly rank deficient (sigma_min/sigma_max
    of the conv2_2 patches here: 1e-3), so the pseudo-inverses of the next stage amplify the differences of the
    previous one by about that ratio (measured: 1e-7 -> 3.5e-5 with exact-product statistics, 3e-6 -> 1e-2 with the
    tensor-core ones; the stage-by-stage test above bounds each stage's own deviation at 3e-6 in both).  Individual
    weights are therefore compared loosely; what must hold is what the reference guarantees -- the discrete outcome
    (selections, alpha schedule, RNG draws) and the function the network computes."""
    from cpb200.lib import cfgs

    spec, g, net, images = _frozen_net(engine, golden_dir, name, mode)
    WPQ, new_pt = net.R3()
    assert cfgs.alpha == float(g["alpha_final"])
    assert np.random.randint(0, 1 << 30) == int(g["rng_after"])
    for k in [k for k in g if k.startswith("sel__")]:
        assert np.array_equal(net.selection[k[5:]], g[k]), k
    _, specs, _, _ = cases.r3_inputs(**spec["gen"])

    def forward(weights, biases):
        x = images[0]
        for s in specs:
            if s.get("type") == "pool":
                B, c, H, W = x.shape
                x = x[:, :, :H // 2 * 2, :W // 2 * 2].reshape(B, c, H // 2, 2, W // 2, 2).max((3, 5))
            else:
                x = np.maximum(O.conv2d_numpy(x, weights[s["name"]], biases[s["name"]], s["pad"], s["stride"]), 0)
        return x

    live = forward({k: v.cpu().numpy() for k, v in net._w.items()}, {k: v.cpu().numpy() for k, v in net._b.items()})
    ref = forward({k[3:]: g[k] for k in g if k.startswith("w__")}, {k[3:]: g[k] for k in g if k.startswith("b__")})
    e_out = float(np.linalg.norm(live - ref) / np.linalg.norm(ref))
    worst = 0.0
    for k in [k for k in g if k.startswith("w__")]:
        worst = max(worst, float(np.linalg.norm(net._w[k[3:]].cpu().numpy() - g[k]) / np.linalg.norm(g[k])))
    print("R3 %s mode %d free running: network output deviates %.2e, worst weight tensor %.2e" % (name, mode, e_out, worst))
    assert e_out <= (1e-3 if mode == 0 else 2e-2) and worst <= (1e-3 if mode == 0 else 5e-2)


def test_frozen_pickle_round_trip(engine, tmp_path):
    """freeze_images writes [feats_dict, points_dict] with protocol 4 (net.py:799-800); load_frozen(DEBUG=True)
    re-extracts at the frozen points and must reproduce the frozen features exactly (net.py:866-875)."""
    from cpb200.lib import cfgs
    from cpb200.lib import net as cpnet

    spec = cases.R3_CASES["r3_small"]
    path = str(tmp_path / "frozen.pickle")
    net, images = build_net(engine, spec, cpnet.ConvStackForward, frozen=path)
    cfgs.c.nBatches, cfgs.c.nPointsPerLayer = 6, 5
    np.random.seed(3)
    assert net.freeze_images() == path
    with open(path, "rb") as f:
        feats_dict, points_dict = pickle.load(f)
    assert set(feats_dict) == set(net.convs) and feats_dict["conv1_1"].dtype == np.float64
    assert feats_dict["conv1_1"].shape == (6 * 5 * images[0].shape[0], 12)
    assert points_dict["nBatches"] == 6 and points_dict["nPointsPerLayer"] == 5 and points_dict["data"] == images[0].shape
    assert points_dict[(2, "conv2_1", "randx")].shape == (5,) and points_dict[(5, 0)].shape == images[0].shape
    net2, _ = build_net(engine, spec, cpnet.ConvStackForward, frozen=path)
    net2.load_frozen(DEBUG=True)
    assert net2.freeze_images(check_exist=True) == path
