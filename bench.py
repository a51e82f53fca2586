#!/usr/bin/env python
"""Headline benchmark: conv layers pruned per second on synthetic VGG-16 conv stacks
(BASELINE.json configs[1]: 13 layers, N=5000 sampled 3x3 patches per layer, random-init weights).

    python bench.py --gpus 1 --steps K --warmup W
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # the CPU restatement of the reference, same metric
    python bench.py --workload sweep          # BASELINE configs[4]: N in {1k,5k,20k,100k} on the conv4_3 shape
    python bench.py ... --dump-outputs DIR    # also writes the results of the last timed step as DIR/*.npy

One "step" = the whole hot path (sparse-point im2col -> Gram statistics -> LASSO channel
selection -> least-squares reconstruction) over one pool of layer problems.

value : layers/s with the feature maps already resident in HBM (device timed, max over ranks).  WEAK scaling: at N
        GPUs the pool holds N networks (13*N independent layer problems) assigned to ranks by LPT, and every step
        ends with the single all_gather that re-assembles the pruned weight dict on all ranks.
strong: (N > 1, extra object) ONE network's 13 problems split over the N GPUs -- north_star's sharding; bounded by
        the critical path of the largest layer, reported with the per-rank device times.
e2e   : the weak metric with feature maps in pinned HOST memory (H2D inside the timed region) and the results copied
        back to the host.
parity: every run checks its own output: two of the timed layer problems are re-solved by the CPU oracle on the
        same arrays (mask, alpha-probe sequence, weights, bias).
Inputs per step (~18 GB of feature maps per network) are far larger than the 126 MB L2, so no L2
flush is needed between timed iterations of the step; the stand-alone kernel timings for the
rooflines flush L2 explicitly.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "conv_layers_pruned_per_sec"
UNIT = "layers/s"
WORKLOADS = {"vgg16": "vgg16_conv_stack_13_layers_N5000", "resnet50": "resnet50_bottlenecks_48_problems_N5000",
             "sweep": "conv4_3_patch_count_sweep_N1k_5k_20k_100k"}
PARITY_LAYERS = {"vgg16": ("conv2_2", "conv3_2"), "resnet50": ("res3b_branch2b", "res4b_branch2a")}


def workload_shapes(args):
    import cpb200

    shapes = cpb200.synth.vgg16_layers() if args.workload == "vgg16" else cpb200.synth.resnet50_layers()
    return select_shapes(shapes, args.layers)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cpb200", choices=["cpb200", "reference"])
    ap.add_argument("--streams", type=int, default=13)
    ap.add_argument("--gram", default="tc", choices=["tc", "fp64"],
                    help="arithmetic of the big Gram products: tc = tcgen05 3xTF32 (default), fp64 = DFMA")
    ap.add_argument("--layout", default="nhwc", choices=["nhwc", "nchw"],
                    help="HBM layout of the bottom blobs for the device-resident arm (nhwc: TMA gather; the host copies of "
                         "the e2e arm keep the reference's NCHW blob order)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="N > 1: skip the strong-scaling leg")
    ap.add_argument("--layers", default="", help="comma list of layer names (debug); default: all of the workload")
    ap.add_argument("--workload", default="vgg16", choices=["vgg16", "resnet50", "sweep"],
                    help="vgg16 = BASELINE configs[1] (13 conv layers); resnet50 = configs[3] (48 bottleneck problems); "
                         "sweep = configs[4] (Gram roofline and LASSO data-form kernel against N)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (see dump_outputs); "
                         "the inputs are seeded, so two builds run with the same arguments can be compared file by file")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl != "cpb200" or args.workload == "sweep"):
        ap.error("--dump-outputs needs the GPU arm of the vgg16 or resnet50 workload")
    return args


def config_dict(args, base, world):
    """Identical for both arms (the driver compares them)."""
    return {"workload": WORKLOADS[args.workload], "layers_per_network": len(base), "networks": world,
            "N_patches": base[0].N,
            "l2": "inputs (feature maps, ~%.1f GB per network) exceed L2; no flush needed"
                  % (sum(4.0 * s.N // (s.B * s.P) * s.B * s.c * s.H * s.W for s in base) / 1e9)}


# ------------------------------------------------------------------------------ CPU arm (oracle)
def shape_classes(shapes):
    """One representative per distinct (c, n, k) -- CPU cost does not depend on the map size."""
    classes = {}
    for s in shapes:
        classes.setdefault((s.c, s.n, s.k), []).append(s)
    return classes


def oracle_on_arrays(shape, fmap, randx, randy, W2, b2, feats, samples, seeds, form="dense"):
    """Runs the oracle (restated reference: numpy patch gather + sklearn-faithful LASSO search + gelsd least squares,
    float64) on one layer problem given as host arrays.  Returns (idxs, W, B, info) with info['t_*'] phase seconds."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np

    import cp_oracle as O

    pd = {"nPointsPerLayer": shape.P, "nBatches": shape.nbatch}
    for b in range(shape.nbatch):
        pd[(b, "y", "randx")] = randx[b]
        pd[(b, "y", "randy")] = randy[b]
    forward = lambda b: {"x": fmap[b * shape.B:(b + 1) * shape.B]}  # noqa: E731
    spec = O.ConvSpec("y", "x", shape.k, shape.pad, shape.stride)
    info = {}
    st = O.DictState(alpha=1e-3)
    rng = O.SeedFeeder(seeds) if seeds is not None else None
    idxs, W, B = O.dictionary_kernel(forward, "x", spec, W2, b2, np.asarray(feats, dtype=np.float64), pd, shape.rank,
                                     state=st, samples=samples, form=form, info=info, rng=rng)
    return idxs, W, B, info


def cpu_layer_seconds(shape, seed):
    """Times the oracle on one synthetic layer problem.  Returns (seconds, phase dict)."""
    import cpb200

    d = cpb200.synth.make_problem_numpy(shape, seed)
    t0 = time.perf_counter()
    _, _, _, info = oracle_on_arrays(shape, d["fmap"], d["randx"], d["randy"], d["W2"], d["b2"], d["feats"], d["samples"],
                                     None)
    return time.perf_counter() - t0, {k: info.get(k, 0.0) for k in ("t_gather", "t_lasso", "t_ls")}


def class_rep(members):
    """The class member with the smallest map (identical solver work, less host memory for the maps), capped at
    28x28: a 224x224x64-channel map set is 6.4 GB of host RAM and ~20 s of random-number generation per layer."""
    import cpb200

    rep = min(members, key=lambda s: s.H)
    return cpb200.synth.LayerShape(rep.name, rep.c, rep.n, min(rep.H, 28), k=rep.k, pad=rep.pad, stride=rep.stride,
                                   N=rep.N, B=rep.B, P=rep.P, rank=rep.rank)


def stack_rate(shapes, cache):
    classes = shape_classes(shapes)
    total = sum(cache[key]["s"] * len(members) for key, members in classes.items())
    return len(shapes) / total


def cpu_full_pass(shapes, cache):
    """One problem per shape class (cost-ascending), stored in cache[class] = {s, phases, n}."""
    classes = shape_classes(shapes)
    t0 = time.perf_counter()
    for key in sorted(classes, key=lambda k: k[0] * k[0] * k[1]):
        t, ph = cpu_layer_seconds(class_rep(classes[key]), 900 + sorted(classes).index(key))
        cache[key] = {"s": t, "phases": ph, "n": 1}
    return time.perf_counter() - t0


def host_threads():
    try:
        from threadpoolctl import threadpool_info

        n = max([p.get("num_threads", 1) for p in threadpool_info()] + [1])
        return int(n)
    except Exception:
        return os.cpu_count() or 1


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host core."""
    n = os.cpu_count() or 1
    try:
        from threadpoolctl import threadpool_limits

        threadpool_limits(limits=n)
    except Exception:
        pass
    return n


REF_BUDGET_S = 165.0
SAMPLE_DESC = ("one layer problem per distinct (c,n,k) class of the stack (feature maps capped at 28x28: solver work "
               "is independent of the map size and a full-size conv1_2 map set alone is 6.4 GB of host RAM), "
               "value = layers / sum(class multiplicity x class seconds)")


def run_reference(args):
    """CPU arm.  A step is a BOUNDED sample: one class problem of the stack (classes visited round-robin in
    cost-ascending order; a class whose last timing no longer fits the run budget is skipped in favour of the most
    expensive one that does).  ms_per_step is the measured mean wall time of the timed steps -- what was run --;
    value extrapolates the classes' mean seconds to the 13-layer stack by multiplicity (stated in `sample`)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ncores = use_all_host_threads()
    shapes = workload_shapes(args)
    classes = shape_classes(shapes)
    order = sorted(classes, key=lambda k: k[0] * k[0] * k[1])
    cache, t_run = {}, time.perf_counter()
    nsteps = max(1, args.steps)
    todo = args.warmup + nsteps
    step_secs, timed_layers = [], 0
    for it in range(todo):
        left = REF_BUDGET_S - (time.perf_counter() - t_run)
        key = order[it % len(order)]
        if key in cache and cache[key]["s"] > left / max(1, todo - it):
            fits = [k for k in order if k not in cache or cache[k]["s"] <= left / max(1, todo - it)]
            key = fits[-1] if fits else order[0]
        t0 = time.perf_counter()
        t, ph = cpu_layer_seconds(class_rep(classes[key]), 900 + sorted(classes).index(key) + 17 * it)
        c = cache.setdefault(key, {"s": 0.0, "phases": {k: 0.0 for k in ph}, "n": 0})
        c["s"] = (c["s"] * c["n"] + t) / (c["n"] + 1)
        for k in ph:
            c["phases"][k] = (c["phases"][k] * c["n"] + ph[k]) / (c["n"] + 1)
        c["n"] += 1
        if it >= args.warmup:
            step_secs.append(time.perf_counter() - t0)
            timed_layers += 1
    missing = [k for k in order if k not in cache]
    for key in missing:  # fewer steps than classes: the estimate still needs every class once
        t, ph = cpu_layer_seconds(class_rep(classes[key]), 900 + sorted(classes).index(key))
        cache[key] = {"s": t, "phases": ph, "n": 1}
    v = stack_rate(shapes, cache)
    phases = {k: sum(cache[key]["phases"][k] * len(m) for key, m in classes.items()) for k in ("t_gather", "t_lasso", "t_ls")}
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * statistics.mean(step_secs), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(args, shapes, max(1, args.gpus)),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": ncores, "blas_threads": host_threads(), "kind": "port",
                         "sample": SAMPLE_DESC + "; a step = ONE class problem (round-robin, cost-ascending; classes that "
                         "no longer fit the %.0f s run budget keep their earlier timing); %d problems in %d timed steps%s"
                         % (REF_BUDGET_S, timed_layers, nsteps,
                            "; %d classes timed once outside the steps" % len(missing) if missing else ""),
                         "stack_seconds": {"gather": phases["t_gather"], "lasso": phases["t_lasso"], "ls": phases["t_ls"]},
                         "class_seconds": {"%dx%dk%d" % k: round(cache[k]["s"], 3) for k in order},
                         "note": "CPU restatement of lib/net.py + lib/decompose.py (oracle port: numpy + C coordinate "
                                 "descent following sklearn _cd_fast.pyx, LAPACK gelsd); the Python reference itself "
                                 "cannot travel to the GPU box",
                         "env": {k: os.environ.get(k) for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS")}},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------ helpers
def select_shapes(shapes, layers):
    if not layers:
        return shapes
    want = set(layers.split(","))
    return [s for s in shapes if s.name in want]


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def ncu_traffic():
    """DRAM bytes per launch of the dominant kernels from the committed ncu --set full captures (profiles/)."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(p):
        return json.load(open(p))
    return {}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


def library_peaks(torch, dev):
    """cuBLAS TF32 and FP64 GEMM throughput on THIS box (denominators only; MEASURED_PEAKS.json holds bf16 and HBM).
    Burst figures: best of 5 after warm-up, CUDA events."""
    out = {}
    old = torch.backends.cuda.matmul.allow_tf32
    try:
        for name, n, dt, tf32 in (("tf32_tflops", 8192, torch.float32, True), ("fp64_tflops", 4096, torch.float64, False)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            a = torch.randn(n, n, device=dev, dtype=dt)
            b = torch.randn(n, n, device=dev, dtype=dt)
            best = 1e9
            for it in range(7):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                torch.matmul(a, b)
                e1.record()
                torch.cuda.synchronize()
                if it >= 2:
                    best = min(best, e0.elapsed_time(e1))
            out[name] = 2.0 * n ** 3 / (best / 1e3) / 1e12
            del a, b
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    return out


def timed_alone(torch, dev, fn, reps=6, skip=2):
    """Mean CUDA-event time (ms) of fn() run alone with an L2 flush before every repetition."""
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    times = []
    for it in range(reps):
        flush.fill_(it)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        if it >= skip:
            times.append(a.elapsed_time(b))
    return statistics.mean(times)


def parity_check(shapes, datas, results, names):
    """Re-solves the named layer problems with the CPU oracle on the SAME arrays the GPU just used and compares."""
    import numpy as np

    import cpb200

    out = {"layers_checked": [], "mask_equal": True, "probes_equal": True, "rel_W_max": 0.0, "rel_b_max": 0.0,
           "oracle": "cp_oracle.dictionary_kernel (sklearn data-form coordinate descent restated in C, LAPACK gelsd)",
           "tolerance": {"rel_W": 1e-4, "rel_b": 1e-4}}
    for s, d, r in zip(shapes, datas, results):
        if s.name not in names or s.name in out["layers_checked"]:
            continue
        t0 = time.perf_counter()
        oi, oW, oB, info = oracle_on_arrays(s, cpb200.synth.fmap_nchw(d).contiguous().cpu().numpy(), d["randx"].cpu().numpy(), d["randy"].cpu().numpy(),
                                            d["W2"].cpu().numpy(), d["b2"].cpu().numpy(), d["feats"].cpu().numpy(),
                                            d["samples"].cpu().numpy(), d["seeds"])
        W = (r.W if not r.W.is_cuda else r.W.cpu()).numpy().reshape(-1)
        b = (r.b if not r.b.is_cuda else r.b.cpu()).numpy()
        same = bool(np.array_equal(r.idxs, oi))
        out["mask_equal"] &= same
        if r.probes is not None:
            plog = r.probes.probe_log[:r.nprobe].cpu().numpy()
            out["probes_equal"] &= [(float(a), int(z)) for a, z, _, _ in plog] == info["probes"]
        if same:
            out["rel_W_max"] = max(out["rel_W_max"], float(np.linalg.norm(W - oW.reshape(-1)) / np.linalg.norm(oW)))
            out["rel_b_max"] = max(out["rel_b_max"], float(np.abs(b - oB).max() / max(1.0, np.abs(oB).max())))
        out["layers_checked"].append(s.name)
        out.setdefault("oracle_seconds", {})[s.name] = round(time.perf_counter() - t0, 2)
    out["pass"] = bool(out["layers_checked"] and out["mask_equal"] and out["probes_equal"] and
                       out["rel_W_max"] <= 1e-4 and out["rel_b_max"] <= 1e-4)
    return out


DUMP_W_BYTES = 56 << 20  # all W files together; masks, biases and the two scalar arrays take well under 8 MB more


def dump_outputs(out_dir, indices, shapes, results):
    """Writes the results of one step of the pool (problem i of the pool is prefixed %03d): <i>_<layer>_mask (kept input
    channels, float32 0/1), <i>_<layer>_W and <i>_<layer>_b (reconstructed weights and bias, float64), and alpha /
    nprobe (the accepted alpha and the number of probes of every problem, in pool order).  A layer whose W could exceed
    its share of DUMP_W_BYTES is sampled by output channel: the rows are a fixed seeded draw that depends only on the
    layer's shape, never on the outputs, so two builds store the same rows."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    cap = DUMP_W_BYTES // 8 // len(results)  # fp64 values of W per problem
    for i, s, r in zip(indices, shapes, results):
        name = os.path.join(out_dir, "%03d_%s_" % (i, s.name))
        W = r.W.cpu().numpy().reshape(s.n, -1)
        if s.n * s.K > cap:  # s.K columns if every input channel were kept
            W = W[np.sort(np.random.RandomState(i).choice(s.n, max(1, cap // s.K), replace=False))]
        np.save(name + "mask.npy", np.asarray(r.idxs, dtype=np.float32))
        np.save(name + "W.npy", W.astype(np.float64))
        np.save(name + "b.npy", r.b.cpu().numpy().astype(np.float64))
    np.save(os.path.join(out_dir, "alpha.npy"), np.array([r.alpha for r in results], dtype=np.float64))
    np.save(os.path.join(out_dir, "nprobe.npy"), np.array([r.nprobe for r in results], dtype=np.float64))


# ------------------------------------------------------------------------------ GPU arm
def run_gpu(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import cpb200
    from cpb200 import pruner

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    eng = cpb200.Engine(device=local, nstreams=args.streams,
                        gram_mode=cpb200.engine.GRAM_3XTF32 if args.gram == "tc" else cpb200.engine.GRAM_FP64)
    lib = cpb200._cabi.load()[1]
    dev = eng.device

    base = workload_shapes(args)
    shapes = [s for _ in range(world) for s in base]  # one network per GPU in the pool (weak scaling)
    owner = pruner.assign_layers([s.cost() for s in shapes], world)
    mine = [i for i, o in enumerate(owner) if o == rank]
    my_shapes = [shapes[i] for i in mine]
    want_e2e = not args.no_e2e
    e2e_skip = None
    if want_e2e:
        # the e2e leg keeps every owned feature map in pinned host memory (18 GB per VGG-16 network and rank):
        # refuse up front, on every rank alike, rather than die inside cudaHostAlloc on a small host
        need = max(sum(shapes[i].nbatch * shapes[i].B * shapes[i].c * shapes[i].H * shapes[i].W * 4
                       for i in range(len(shapes)) if owner[i] == r) for r in range(world)) * world
        try:
            import psutil
            avail = psutil.virtual_memory().available
        except Exception:  # pragma: no cover
            avail = None
        if world > 1:  # one decision for all ranks (they probe at slightly different times): the smallest view wins
            t = torch.tensor([float(avail if avail is not None else 1e18)], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            avail = None if t.item() >= 1e18 else t.item()
        if avail is not None and need > 0.6 * avail:
            want_e2e = False
            e2e_skip = "host has %.0f GB available, the pinned feature maps of %d ranks need %.0f GB" % (
                avail / 1e9, world, need / 1e9)
    # the pinned host copies of the e2e leg are made AFTER the device-resident measurement: they are no input of it
    datas = [cpb200.synth.make_problem_device(shapes[i], 1000 + i, eng, pinned_host=False, layout=args.layout)
             for i in mine]
    sizes = [pruner.slot_size(s.c, s.n, s.k * s.k, s.rank, .1) for s in shapes]
    per_rank = [sum(sizes[i] for i in range(len(shapes)) if owner[i] == r) for r in range(world)]
    gbuf = torch.zeros(max(per_rank), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()

    def step(from_host, shp=my_shapes, dat=datas, idx=mine, all_shapes=shapes, all_sizes=sizes):
        res = pruner.prune_layers(eng, shp, dat, right0=1e-3, rank_tol=.1, from_host=from_host, to_host=from_host)
        if world > 1:
            off = 0
            for j, i in enumerate(idx):
                s = all_shapes[i]
                pruner.pack_result(gbuf, off, res[j].idxs, res[j].W, res[j].b, res[j].alpha, res[j].nprobe, s.c, s.n,
                                   s.k * s.k, eng=eng, slot=j)
                off += all_sizes[i]
            pruner.allgather_results(gbuf, world)
        return res

    def timed(nsteps, fn):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = lib.cp_launch_count()
        t_host = time.perf_counter()
        e0.record()
        res = None
        for _ in range(nsteps):
            res = fn()
        e1.record()
        host_issue = time.perf_counter() - t_host  # host time spent ISSUING the steps (incl. the mask read-backs)
        torch.cuda.synchronize()
        ms_local = e0.elapsed_time(e1)
        ms = ms_local
        launches = lib.cp_launch_count() - l0
        per_rank_ms = [ms_local]
        if world > 1:
            t = torch.tensor([ms_local], device=dev, dtype=torch.float64)
            allt = torch.empty(world, device=dev, dtype=torch.float64)
            dist.all_gather_into_tensor(allt, t)
            per_rank_ms = [float(x) for x in allt.cpu()]
            ms = max(per_rank_ms)
            dist.barrier()
        return ms, launches, res, host_issue, per_rank_ms

    for _ in range(args.warmup):
        step(False)
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms, launches, res, host_issue, _ = timed(args.steps, lambda: step(False))
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:  # before any later leg reuses the engine's buffers
        dump_outputs(args.dump_outputs, mine, my_shapes, res)
    total_layers = len(shapes) * args.steps
    value = total_layers / (ms / 1e3)

    parity = None
    if rank == 0 and not args.no_parity:
        parity = parity_check(my_shapes, datas, res, PARITY_LAYERS.get(args.workload, ()))
    ls_paths = {}
    for s, r in zip(my_shapes, res):
        ls_paths[r.info.get("verdict", "?")] = ls_paths.get(r.info.get("verdict", "?"), 0) + 1
    min_ratio = min([r.info.get("pivot_ratio", 1.0) for r in res] + [1.0])

    e2e = None
    if want_e2e:
        for d in datas:  # the reference's blob order (NCHW) in page-locked host memory
            src = cpb200.synth.fmap_nchw(d)
            with cpb200.engine.numa_local(local):  # pages on the socket this rank's GPU hangs off
                d["fmap_host"] = torch.empty(src.shape, dtype=torch.float32, pin_memory=True)
                d["fmap_host"].copy_(src)
        torch.cuda.synchronize()
        for _ in range(min(args.warmup, 3)):
            step(True)
        ms_e, _, res_e, _, _ = timed(args.steps, lambda: step(True))
        # the feature maps stay in pinned host memory; per layer either the gather kernel pulls the sampled
        # k x k x c windows over PCIe in place (bytes that must cross: 4*N*K) or, where the windows cover most of
        # the map (conv5_x), the copy engine moves the whole map (bytes: the map) -- pruner.h2d_plan decides
        plan = pruner.h2d_plan(my_shapes, datas, True)
        h2d = sum(int(d["fmap_host"].numel()) * 4 if p == "dma" else int(s.N) * s.K * 4
                  for s, d, p in zip(my_shapes, datas, plan))
        host_resident = sum(int(d["fmap_host"].numel()) * 4 for d in datas)
        d2h = sum(int(r.W.numel() + r.b.numel()) * 8 + s.c + 32 for r, s in zip(res_e, my_shapes))
        if world > 1:
            t = torch.tensor([h2d, d2h], device=dev, dtype=torch.float64)
            dist.all_reduce(t)
            h2d, d2h = int(t[0].item()), int(t[1].item())
        e2e = {"value": total_layers / (ms_e / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "ms_per_step": ms_e / args.steps, "host_resident_input_bytes": host_resident,
               "h2d_plan": "".join("D" if p == "dma" else "z" for p in plan),
               "input_path": "feature maps in pinned host memory; per layer (h2d_plan, z/D) read in place by "
                             "cp_patch_gather (zero-copy over PCIe, bytes = gathered windows) or DMA'd whole (bytes = map)"}

    # ---- strong scaling (north_star's split): ONE network's problems over the N GPUs
    strong = None
    if world > 1 and not args.no_strong:
        s_owner = pruner.assign_layers([s.cost() for s in base], world)
        s_mine = [i for i, o in enumerate(s_owner) if o == rank]
        s_shapes = [base[i] for i in s_mine]
        have = {i: d for i, d in zip(mine, datas)}
        s_datas = [have[i] if i in have else cpb200.synth.make_problem_device(base[i], 1000 + i, eng, layout=args.layout)
                   for i in s_mine]
        s_sizes = [pruner.slot_size(s.c, s.n, s.k * s.k, s.rank, .1) for s in base]

        def sstep():
            return step(False, s_shapes, s_datas, s_mine, base, s_sizes)

        for _ in range(max(2, args.warmup // 2)):
            sstep()
        ms_s, _, _, _, per_rank_ms = timed(args.steps, sstep)
        strong = {"value": len(base) * args.steps / (ms_s / 1e3), "unit": UNIT, "ms_per_step": ms_s / args.steps,
                  "networks": 1, "scaling": "strong",
                  "per_rank_ms_per_step": [round(x / args.steps, 3) for x in per_rank_ms],
                  "layers_per_rank": [sum(1 for o in s_owner if o == r) for r in range(world)],
                  "note": "one network split by LPT; the step cannot be shorter than the critical path of its largest "
                          "layer (gather + Gram -> LASSO search -> least squares)"}

    # ---- rooflines of the two kernels north_star names, each timed alone after an L2 flush
    roof = roof_g = None
    peaks_lib = None
    if rank == 0:
        peaks, which = measured_peaks()
        peaks_lib = library_peaks(torch, dev)
        traffic = ncu_traffic()
        s = max(base, key=lambda q: q.K)
        names = [shapes[i].name for i in mine]
        d = datas[names.index(s.name)] if s.name in names else cpb200.synth.make_problem_device(s, 5, eng, layout=args.layout)
        lay = d.get("layout", "nchw")
        X = eng.patch_gather(d["fmap"], d["randx"], d["randy"], s.B, s.P, s.k, s.pad, s.stride, relu=True, layout=lay)
        fp64_mode = eng.gram_mode == cpb200.engine.GRAM_FP64
        gen1 = os.environ.get("CPB200_GRAM_TC", "") == "1"
        kern_ms = []
        t_ms = timed_alone(torch, dev, lambda: eng.gram(X, d["feats"], y_bias=d["b2"], want_sums=False))
        if not fp64_mode and not gen1:
            # second pass with CUDA events around the tcgen05 GEMM launch (on its stream), read after each call
            eng.gram_profile(True)

            def one_gram():
                eng.gram(X, d["feats"], y_bias=d["b2"], want_sums=False)
                kern_ms.append(eng.gram_kernel_ms())

            timed_alone(torch, dev, one_gram)
            eng.gram_profile(False)
        flops = float(s.N) * s.K * (s.K + 1) + 2.0 * s.N * s.K * s.n  # SURVEY.md 8(d): symmetric half + X'Y
        call_tflops = flops / (t_ms / 1e3) / 1e12
        if fp64_mode:
            kernel, k_ms = "cp_gram (fp64 products)", t_ms
            peak, peak_note = peaks_lib["fp64_tflops"], "cuBLAS FP64 GEMM 4096^3 measured in this run"
            extra = {}
        elif gen1:
            kernel, k_ms = "cp_gram, first-generation gram_tc_kernel (3xTF32) + its passes", t_ms
            peak, peak_note = peaks_lib["tf32_tflops"], "cuBLAS TF32 GEMM 8192^3 measured in this run; 3 MMAs per product: ceiling 1/3"
            extra = {}
        else:
            # the dominant kernel of the call, timed alone: gram_tc2_pair_kernel (kind::f16 tcgen05, three products of
            # the split-fp16 operands per algorithmic product -> ceiling = 1/3 of the dense 16-bit rate)
            k_ms = sum(kern_ms[2:]) / max(1, len(kern_ms[2:]))
            kernel = "gram_tc2_pair_kernel (tcgen05 kind::f16, cta_group::2, 256x256 tiles; 3 MMAs per product)"
            peak = peaks["bf16_tflops"]
            peak_note = "dense bf16 burst of MEASURED_PEAKS.json (%s); split-precision scheme issues 3 MMAs per " \
                        "algorithmic product: ceiling 1/3" % which
            extra = {"issued_tflops": 3.0 * flops / (k_ms / 1e3) / 1e12, "frac_issued": 3.0 * flops / (k_ms / 1e3) / 1e12 / peak,
                     "call": {"what": "whole cp_gram call (statistics passes, operand preparation, GEMM, fp64 reduction "
                                      "of the splits, lower triangle)", "ms": t_ms, "achieved": call_tflops,
                              "frac": call_tflops / peak},
                     "cublas_tf32_tflops": peaks_lib["tf32_tflops"]}
        achieved = flops / (k_ms / 1e3) / 1e12
        tr = traffic.get("gram_tc2_pair_kernel" if not gen1 else "gram_tc_kernel") if not fp64_mode else None
        roof = {"kernel": "%s on %s: N=%d K=%d n=%d (X'X upper tiles + X'Y)" % (kernel, s.name, s.N, s.K, s.n),
                "bound": "tensor" if not fp64_mode else "fp64-pipe",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "traffic": tr["bytes"] if tr and s.name == "conv4_2" and s.N == 5000 else None,
                "traffic_source": tr["source"] if tr else None,
                "ms": k_ms, "algorithmic_flops": flops, "peak_source": peak_note,
                "mode": "fp64" if fp64_mode else ("3xtf32" if gen1 else "3xfp16-split")}
        roof.update(extra)
        t_g = timed_alone(torch, dev, lambda: eng.patch_gather(d["fmap"], d["randx"], d["randy"], s.B, s.P, s.k, s.pad,
                                                               s.stride, relu=True, out=X, layout=lay))
        gbytes = 8.0 * s.N * s.K  # SURVEY.md 8(d): unique patch elements read + X written
        trg = traffic.get("patch_gather_nhwc_tma" if lay == "nhwc" else "patch_gather")
        # the other layout, for the record (same values, same X)
        fm_other = cpb200.synth.fmap_nchw(d).contiguous() if lay == "nhwc" else d["fmap"].permute(0, 2, 3, 1).contiguous()
        other = "nchw" if lay == "nhwc" else "nhwc"
        X2 = torch.empty_like(X)
        t_o = timed_alone(torch, dev, lambda: eng.patch_gather(fm_other, d["randx"], d["randy"], s.B, s.P, s.k, s.pad,
                                                               s.stride, relu=True, out=X2, layout=other))
        same_X = bool(torch.equal(X, X2))
        del fm_other, X2
        roof_g = {"kernel": "cp_patch_gather (sparse-point im2col, %s%s) on %s: N=%d K=%d" % (
                      lay.upper(), ", TMA window loads + bulk row stores" if lay == "nhwc" else "", s.name, s.N, s.K),
                  "other_layout": {"layout": other, "ms": t_o, "GB/s": gbytes / (t_o / 1e3) / 1e9, "X_bit_identical": same_X},
                  "bound": "hbm", "achieved": gbytes / (t_g / 1e3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                  "frac": gbytes / (t_g / 1e3) / 1e9 / peaks["hbm_gbs"],
                  "traffic": trg["bytes"] if trg else None, "traffic_source": trg["source"] if trg else None,
                  "ms": t_g, "algorithmic_bytes": gbytes, "peak_source": "%s copy bandwidth (MEASURED_PEAKS.json)" % which}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        ncores = use_all_host_threads()
        cache = {}
        secs = cpu_full_pass(base, cache)
        classes = shape_classes(base)
        cpu = {"value": stack_rate(base, cache), "unit": UNIT, "cores": ncores, "blas_threads": host_threads(),
               "kind": "port", "sample": SAMPLE_DESC, "seconds": secs,
               "stack_seconds": {k[2:]: sum(cache[key]["phases"][k] * len(m) for key, m in classes.items())
                                 for k in ("t_gather", "t_lasso", "t_ls")}}

    if rank == 0:
        kept = [int(r.idxs.sum()) for r in res]
        cfg = config_dict(args, base, world)
        cfg.update(streams=args.streams, kept_channels_rank0=kept, hbm_layout=args.layout)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64" if eng.gram_mode == cpb200.engine.GRAM_FP64 else "f16x3-split+f64", "data": "synthetic",
            "config": cfg, "clocks": clocks,
            "e2e": e2e if e2e is not None or e2e_skip is None else {"unavailable": e2e_skip},
            "gpu_launches": int(launches // max(1, args.steps)),
            "host_issue_ms_per_step": 1e3 * host_issue / max(1, args.steps),
            "roofline": roof, "roofline_im2col": roof_g, "library_peaks": peaks_lib, "parity": parity,
            "ls_policy": {"paths": ls_paths, "min_pivot_ratio": min_ratio, "ratio_min_for_tc": cpb200.engine.LS_RATIO_MIN},
            "strong": strong, "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.workload == "sweep":
        from profiles import sweep_config5

        sweep_config5.main(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
