#!/usr/bin/env python
"""Benchmark of the sparse-voxel hot path under the reference's segmentors: scans/s of one training step.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config C] [--batch B] [--model-src S]
                    [--dtype fp16|fp32] [--impl ours|reference|reference_cuda]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

One "step" = one training step (AMP fp16 forward + backward + SGD update, as train.py:340-372 of the
reference) over one batch of B synthetic SemanticKITTI-shaped scans (64 x 1875 rays) per GPU.

  --config     minkunet34 (default; BASELINE configs[1], the headline) | spvcnn18 | cylinder480 | rpvnet34
               (BASELINE configs[2..4]); B defaults to the reference yaml's BATCH_SIZE_PER_GPU (16 for the
               headline, as in round 1)
  --model-src  native     openpcseg_b200.segmentors.MinkUNet (same architecture / state_dict, BN+ReLU fused;
                          minkunet34 only, its default)
               reference  the reference's OWN segmentor class, staged unmodified under oracle/_ref/py,
                          running on this backend through install_as_torchsparse() (default for the others)
  --impl       ours            this backend (libb2s) - the line the driver reads
               reference       the reference's own CPU implementation (its segmentor class on the CPU build of its
                               torchsparse, oracle/_ref) on host cores, bounded sub-scan per step, rank 0 only
               reference_cuda  the reference's own CUDA torchsparse recompiled for sm_100a
                               (oracle/build_ref_cuda.py) under the same class, same GPU, same inputs

Prints ONE JSON line:
  value         scans/s over all GPUs, inputs resident in HBM when the timed region starts
  e2e           the same through the public API with pinned HOST buffers: every step's batch is copied host ->
                device (copy stream, one step ahead) and every step's loss device -> host (asynchronously, read by
                the host one step late), all inside the timed region
  roofline      the dominant conv kernel family timed live with CUDA events around every launch, in a
                repeat of the same K steps after the `value` region
  cpu_baseline  the reference's CPU path on a bounded sub-scan (rank 0, N=1)
  ref_cuda      (N=1) the reference's CUDA build on the same workload, measured in the same run by a
                child process of this script (--impl reference_cuda); None when oracle/_ref has no CUDA build
  config1       (N=1) BASELINE configs[0]: one k3 submanifold conv on a 10 k-point cloud - naive PyTorch
                gather-matmul-scatter on the host cores, the reference CPU backend, and this backend
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# per-batch buffer sizes differ (kernel maps, step tables: up to 160 MB each): growable segments keep the caching
# allocator from re-splitting / cudaMalloc-ing inside the timed steps
os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")

import numpy as np  # noqa: E402
import torch  # noqa: E402

FULL_AZIMUTH = 1875
CONFIGS = {
    # name: (batch kind, default scans/GPU/step, metric label, workload label)
    "minkunet34": ("voxel", 16, "scans/s MinkUNet-34 fwd+bwd @~120k pts/0.05 m voxel",
                   "MinkUNet-34 cr1.0 fwd+bwd(+SGD step), synthetic SemanticKITTI 64x1875 rays, 0.05 m voxel"),
    "spvcnn18": ("voxel", 16, "scans/s SPVCNN-18 cr1.0 fwd+bwd @~120k pts/0.05 m voxel",
                 "SPVCNN mk18 cr1.0 fwd+bwd(+SGD step), synthetic SemanticKITTI 64x1875 rays, 0.05 m voxel"),
    "cylinder480": ("cylinder", 12, "scans/s Cylinder3D cy480 fwd+bwd @120k pts/480x360x32 cylinder grid",
                    "Cylinder3D cy480 cr1.0 fwd+bwd(+SGD step), synthetic SemanticKITTI 64x1875 rays, "
                    "480x360x32 cylindrical grid"),
    "rpvnet34": ("fusion", 4, "scans/s RPVNet-34 cr1.75 fwd+bwd @~120k pts/0.05 m voxel + 64x2048 range image",
                 "RPVNet mk34 cr1.75 fwd+bwd(+SGD step), synthetic SemanticKITTI 64x1875 rays, 0.05 m voxel, "
                 "5x64x2048 range image"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=12)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--config", default="minkunet34", choices=list(CONFIGS))
    ap.add_argument("--batch", type=int, default=int(os.environ.get("B2S_BENCH_BATCH", 0)),
                    help="scans per GPU per step (0 = the config's default)")
    ap.add_argument("--model-src", default=None, choices=["native", "reference"])
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference_cuda"])
    ap.add_argument("--dtype", default="fp16", choices=["fp16", "fp32"])
    ap.add_argument("--sync-bn", action="store_true")
    ap.add_argument("--sm-reserve", type=int, default=None,
                    help="SMs kept free of the persistent conv grids (default 0: measured at N = 2, reserving 8 / 16 "
                         "SMs for NCCL LOSES 3 %% - the all-reduce is not what limits scaling, profiles/r2_scaling.txt)")
    ap.add_argument("--pool", type=int, default=4, help="distinct batches cycled per rank")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-cuda", action="store_true")
    ap.add_argument("--no-config1", action="store_true")
    ap.add_argument("--bucket-mb", type=int, default=1024,
                    help="DDP bucket_cap_mb.  Default: ONE bucket = the gradient all-reduce runs after backward "
                         "instead of under it: NCCL's CTAs otherwise take SM slots from the persistent conv grids, "
                         "whose statically striped CTAs then finish in a second wave (N = 8: 0.89 -> see profiles/)")
    ap.add_argument("--same-data", action="store_true",
                    help="diagnostic: every rank gets rank 0's scans (separates load imbalance from communication)")
    ap.add_argument("--cpu-budget-s", type=float, default=None,
                    help="CPU seconds for the reference arm (default 150 for --impl reference, 25 for the "
                         "cpu_baseline leg of the default run)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, take the timed step once more on the last timed step's batch from "
                         "the run's starting state and write what it computed as DIR/<name>.npy (float32 / float64, "
                         "fixed seeded samples of the large arrays; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.batch <= 0:
        args.batch = CONFIGS[args.config][1]
    if args.model_src is None:
        args.model_src = "native" if (args.config == "minkunet34" and args.impl == "ours") else "reference"
    if args.model_src == "native" and args.config != "minkunet34":
        ap.error("--model-src native exists for minkunet34 only")
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"hbm_gbs": d["hbm_gbs"], "tflops_burst": d["bf16_tflops"],
                "tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "source": "fallback"}


# ------------------------------------------------------------------ CPU reference arm
def cpu_reference_run(config: str, budget_s: float, steps: int, warmup: int, full_units: int | None = None):
    """Time the reference's OWN segmentor class on the CPU build of its own torchsparse (oracle/_ref; for
    RPVNet / Cylinder3D the CUDA-only range_lib and the absent torch_scatter are torch stand-ins, see
    baseline/loader.py) on a bounded sub-scan; returns (scans_per_s, info dict, ms per step).

    Stock code path of the reference, with two caveats stated in the line: ``Tensor.cuda`` is the identity
    (the models call ``.cuda()`` on the targets) and one scan per step (the reference's CPU kernel-hash
    reads point 0's batch word for every point, TS/backend/hash/hash_cpu.cpp:29)."""
    from baseline import loader
    from openpcseg_b200.synthetic import make_model_batch
    # Thread count: measured on the 128-core B200 host (round 1, 1/32 sub-scan): 8 threads 5.1 s,
    # 32 threads 25.4 s - the reference's per-offset OpenMP gather loops + small MKL GEMMs slow down
    # when oversubscribed, so 8 is its fastest setting.
    cores = min(os.cpu_count() or 1, int(os.environ.get("B2S_CPU_THREADS", 8)))
    torch.set_num_threads(cores)
    os.environ.setdefault("OMP_NUM_THREADS", str(cores))
    kind = CONFIGS[config][0]
    torch.Tensor.cuda = lambda self, *a, **k: self
    ns = loader.activate("ref_cpu")
    torch.manual_seed(0)
    net = ns.build_model(config).train()
    unit_key = "voxel_coord" if kind == "cylinder" else "coords"
    if full_units is None:
        full_units = make_model_batch(kind, [0])[unit_key].shape[0]

    def one(n_az, seed):
        arrays = make_model_batch(kind, [seed], n_azimuth=n_az)
        bd = ns.batch_dict(arrays, "cpu")
        t0 = time.perf_counter()
        ret, _, _ = net(bd)
        ret["loss"].backward()
        net.zero_grad(set_to_none=True)
        return time.perf_counter() - t0, arrays[unit_key].shape[0]

    # calibrate on a 1/32 sub-scan, then size the sample to the time budget
    t_cal, v_cal = one(max(FULL_AZIMUTH // 32, 8), 100)
    rate = v_cal / t_cal                                     # voxels per second, first guess
    per_step = budget_s / max(steps + warmup, 1)
    n_az = int(np.clip(FULL_AZIMUTH * (rate * per_step) / full_units, 24, FULL_AZIMUTH))
    for w in range(warmup):
        one(n_az, 200 + w)
    ts, vs = [], []
    for s in range(steps):
        t, v = one(n_az, 300 + s)
        ts.append(t)
        vs.append(v)
    scans = sum(vs) / full_units                             # fraction-of-scan units processed
    value = scans / sum(ts)
    info = {"value": value, "unit": "scans/s", "cores": cores, "kind": "reference",
            "sample": f"{steps} steps of fwd+bwd of the reference's own {loader.MODELS[config][2]} class on its CPU "
                      f"torchsparse build, one {n_az}/{FULL_AZIMUTH}-azimuth sub-scan per step (~{int(np.mean(vs))} "
                      f"of {full_units} voxels), fp32, scaled by voxel count"}
    return value, info, sum(ts) / max(len(ts), 1) * 1e3


# ------------------------------------------------------- BASELINE configs[0] (10 k-pt k3 conv)
def config1_run(device) -> dict:
    """Single 3x3x3 submanifold conv 16 -> 32 on a 10 k-point cloud U(-10,10)^3 quantised at 0.2 (SURVEY 8d
    config 1), fp32 forward+backward: (i) naive PyTorch gather-matmul-scatter on the host cores,
    (ii) the reference CPU backend, (iii) this backend on the GPU.  ms per call, median of 5."""
    from oracle import build_ref, ref_ops as R
    import openpcseg_b200.torchsparse as ts
    rng = np.random.default_rng(0)
    pts = rng.uniform(-10, 10, size=(10000, 3))
    c = np.unique(np.floor(pts / 0.2).astype(np.int32), axis=0)
    c = np.concatenate([c - c.min(0), np.zeros((len(c), 1), np.int32)], 1).astype(np.int32)
    x = rng.standard_normal((len(c), 16)).astype(np.float32)
    w = (rng.standard_normal((27, 16, 32)) / np.sqrt(27 * 16)).astype(np.float32)
    go = rng.standard_normal((len(c), 32)).astype(np.float32)
    nb, nsz = R.build_kmap(c, c, 3)
    cores = min(os.cpu_count() or 1, int(os.environ.get("B2S_CPU_THREADS", 8)))
    torch.set_num_threads(cores)
    xt, wt, got = torch.from_numpy(x), torch.from_numpy(w), torch.from_numpy(go)
    nbt = torch.from_numpy(nb).long()
    starts = np.concatenate([[0], np.cumsum(nsz)])

    def naive():
        xi, wi = xt.clone().requires_grad_(True), wt.clone().requires_grad_(True)
        out = torch.zeros(len(c), 32)
        for k in range(27):
            p = nbt[starts[k]:starts[k + 1]]
            if len(p):
                out = out.index_add(0, p[:, 1], xi[p[:, 0]] @ wi[k])
        out.backward(got)
        return out

    def med(fn, n=5):
        fn()
        t = []
        for _ in range(n):
            t0 = time.perf_counter()
            fn()
            t.append((time.perf_counter() - t0) * 1e3)
        return statistics.median(t)

    res = {"workload": f"k3 submanifold conv 16->32, {len(c)} voxels, {int(nsz.sum())} pairs, fp32 fwd+bwd",
           "cores": cores, "naive_torch_cpu_ms": med(naive)}
    ref = build_ref.load()
    if ref is not None:
        nb32, ns32 = torch.from_numpy(nb).int(), torch.from_numpy(nsz).int()

        def ref_cpu():
            out = torch.zeros(len(c), 32)
            ref.convolution_forward_cpu(xt, out, wt, nb32, ns32, False)
            gi, gw = torch.zeros_like(xt), torch.zeros_like(wt)
            ref.convolution_backward_cpu(xt, gi, got, wt, gw, nb32, ns32, False)
        res["reference_cpu_backend_ms"] = med(ref_cpu)
    cd, xd, wd, gd = (torch.from_numpy(a).to(device) for a in (c, x, w, go))

    def ours():
        xi, wi = xd.clone().requires_grad_(True), wd.clone().requires_grad_(True)
        st = ts.SparseTensor(xi, cd, 1)
        st.kmaps = kmaps
        st.cmaps[st.stride] = cd
        y = ts.nn.functional.conv3d(st, wi, 3)
        y.feats.backward(gd)
        torch.cuda.synchronize()
    kmaps = {}
    res["this_backend_gpu_ms"] = med(ours)
    return res


# ------------------------------------------------------------------------- helpers
class ConvProfiler:
    """CUDA events around every conv kernel launch of the timed region (events are pre-created so
    that recording them costs ~1 us of host time per launch)."""

    def __init__(self, n_events=0):
        self.rows = []
        self.pool = [torch.cuda.Event(enable_timing=True) for _ in range(n_events)]
        self.next = 0

    def event(self):
        if self.next < len(self.pool):
            ev = self.pool[self.next]
            self.next += 1
            return ev
        return torch.cuda.Event(enable_timing=True)

    def record(self, kind, meta, start, end):
        self.rows.append((kind, meta, start, end))

    def summarise(self):
        out = {}
        totals = {}
        for kind, meta, s, e in self.rows:
            ms = s.elapsed_time(e)
            pairs = meta["pairs"]
            m = int(pairs.item()) if pairs is not None else int(meta["rows"])
            if meta["k"] == 1:
                m = int(meta["rows"])
            flops = 2.0 * m * meta["c_in"] * meta["c_out"]
            e_b = 2 if meta["dtype"] == 1 else 4
            # algorithmic bytes (SURVEY 8d): gathered rows + result rows + map entries + weights
            byts = e_b * meta["c_in"] * m + e_b * meta["c_out"] * meta["rows"] + 8 * m \
                + e_b * meta["k"] * meta["c_in"] * meta["c_out"]
            t = totals.setdefault(kind, [0.0, 0.0, 0, 0.0])
            t[0] += ms
            t[1] += flops
            t[2] += 1
            t[3] += byts
        for k, (ms, fl, n, by) in totals.items():
            out[k] = {"ms": ms, "gflop": fl / 1e9, "launches": n,
                      "tflops": (fl / 1e12) / (ms / 1e3) if ms > 0 else 0.0,
                      "alg_gbs": (by / 1e9) / (ms / 1e3) if ms > 0 else 0.0}
        return out


def clocks_sampler():
    try:
        return subprocess.Popen(
            ["nvidia-smi", "--query-gpu=index,clocks.sm,clocks.max.sm,power.draw,"
             "clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits", "-lms", "100",
             "-i", str(torch.cuda.current_device())],
            stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except Exception:
        return None


def clocks_summary(proc):
    if proc is None:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
    proc.terminate()
    try:
        out, _ = proc.communicate(timeout=5)
    except Exception:
        proc.kill()
        out = ""
    sm, mx, reasons = [], [], set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for line in out.strip().splitlines():
        f = [x.strip() for x in line.split(",")]
        if len(f) < 9:
            continue
        try:
            sm.append(float(f[1]))
            mx.append(float(f[2]))
        except ValueError:
            continue
        for name, val in zip(names, f[5:9]):
            if val.lower().startswith("active"):
                reasons.add(name)
    return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
            "samples": len(sm), "reasons": sorted(reasons)}


DUMP_LOGIT_ROWS = 1 << 18
DUMP_PARAMS = 1 << 20
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(directory: str, out: dict, model: torch.nn.Module) -> dict:
    """Write the results of one training step as ``directory/<name>.npy`` so that two builds run with the same
    arguments (hence the same inputs and initial weights) can be compared array by array:

      loss    float64 [1]       the step's loss
      logits  float32 [R, C]    the step's logits; R = all rows, or a fixed seeded sample of DUMP_LOGIT_ROWS rows
                                (ascending row order) when there are more
      params  float32 [P]       every parameter after the optimizer step, flattened and concatenated in
                                ``model.parameters()`` order; a fixed seeded sample of DUMP_PARAMS elements
                                (ascending index order) when there are more

    The step dumped is the timed step function applied to the batch of the last timed step, starting from the
    model, optimizer and loss-scaler state the run started from (seeded weights, no momentum): the kernels reduce
    with float atomics, so the state reached after the warm-up and timed steps differs from run to run by more
    than the rounding of one step.
    """
    g = torch.Generator().manual_seed(0)

    def sample(n, k):
        return torch.randperm(n, generator=g)[:k].sort().values if n > k else None

    arrays = {"loss": out["loss"].detach().double().cpu().numpy().reshape(1)}
    if "logits" in out:
        y = out["logits"].detach().float()
        rows = sample(y.shape[0], DUMP_LOGIT_ROWS)
        arrays["logits"] = (y if rows is None else y[rows.to(y.device)]).cpu().numpy()
    flat = torch.cat([p.detach().float().reshape(-1) for p in model.parameters()])
    idx = sample(flat.numel(), DUMP_PARAMS)
    arrays["params"] = (flat if idx is None else flat[idx.to(flat.device)]).cpu().numpy()
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_MAX_BYTES
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)
    return {name: list(a.shape) for name, a in arrays.items()}


def ref_cuda_child(args) -> dict | None:
    """Run ``--impl reference_cuda`` of the same config in a child process and return its JSON line."""
    import glob
    if not glob.glob(os.path.join(ROOT, "oracle", "_ref", "ts_ref_backend_cuda.*so")):
        return None
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference_cuda", "--config", args.config,
           "--batch", str(args.batch), "--steps", str(min(args.steps, 6)), "--warmup", "3",
           "--dtype", args.dtype, "--pool", "2", "--no-cpu-baseline"]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
        line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
        d = json.loads(line)
        return {k: d.get(k) for k in ("value", "unit", "ms_per_step", "steps", "e2e", "config", "gpu_launches",
                                       "impl", "dtype")}
    except Exception as exc:                                           # never lose the GPU line
        return {"value": None, "error": f"{type(exc).__name__}: {str(exc)[:200]}"}


def main():
    args = parse()
    from openpcseg_b200 import dist_utils as D
    rank, world, local = D.env_rank_world()
    kind, _, metric, workload = CONFIGS[args.config]

    if args.impl == "reference":
        if rank != 0:
            return
        value, info, ms = cpu_reference_run(args.config, args.cpu_budget_s or 150.0, args.steps, args.warmup)
        line = {"impl": "reference", "metric": metric, "value": value, "unit": "scans/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": workload + " (reference CPU path, bounded sub-scan per step)"},
                "cpu_baseline": info,
                "e2e": {"value": value, "unit": "scans/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    assert torch.cuda.is_available(), "bench.py (impl=ours / reference_cuda) needs a CUDA device"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from openpcseg_b200.synthetic import make_model_batch
    ours = args.impl == "ours"
    B = None
    reserve = 0
    if ours:
        from openpcseg_b200 import backend as B
        # DDP: NCCL's all-reduce kernels need SMs while the backward's persistent grids are resident
        reserve = args.sm_reserve if args.sm_reserve is not None else 0
        B.set_sm_reserve(reserve)

    torch.manual_seed(0)
    amp = args.dtype == "fp16"
    ns = None
    if args.model_src == "native":
        import openpcseg_b200.torchsparse as ts
        from openpcseg_b200.segmentors import MinkUNet, minkunet34_config
        model = MinkUNet(minkunet34_config(sync_bn=args.sync_bn and world > 1)).to(dev)
    else:
        from baseline import loader
        ns = loader.activate("b2s" if ours else "ref_cuda")
        over = {"IF_DIST": True} if (args.sync_bn and world > 1) else {}
        model = ns.build_model(args.config, **over).to(dev)
    model.train()
    net = model
    if world > 1:
        net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local], gradient_as_bucket_view=True,
                                                        bucket_cap_mb=args.bucket_mb)
    # SGD momentum 0.9, weight decay 1e-4 (pcseg/optim/__init__.py:15-21 - the reference never passes
    # NESTEROV on), AMP GradScaler, clip 10 (train.py:367-372); lr is irrelevant to throughput
    # fused=True: torch's multi-tensor SGD kernel takes the GradScaler's found_inf flag ON THE DEVICE, so
    # scaler.step() does not read it back (one host sync per step less; the same optimizer for both arms)
    opt = torch.optim.SGD(model.parameters(), lr=0.01, momentum=0.9, weight_decay=1e-4, fused=True)
    scaler = torch.amp.GradScaler("cuda", enabled=amp)
    start_state = None
    if args.dump_outputs:          # the state the dumped step starts from (see dump_outputs)
        start_state = ({k: v.detach().clone() for k, v in model.state_dict().items()}, opt.state_dict())

    # ---- synthetic data: a pool of distinct batches per rank, in pinned host memory
    unit_key = "voxel_coord" if kind == "cylinder" else "coords"
    pool = []
    for p in range(args.pool):
        seeds = D.scan_seeds(0 if args.same_data else rank, p, args.batch)
        b = make_model_batch(kind, seeds)
        pool.append({k: torch.from_numpy(v).pin_memory() for k, v in b.items() if isinstance(v, np.ndarray)})
    vox_per_scan = float(np.mean([p[unit_key].shape[0] for p in pool])) / args.batch
    h2d = int(np.mean([sum(t.numel() * t.element_size() for t in p.values()) for p in pool]))
    resident = [{k: v.to(dev) for k, v in p.items()} for p in pool]
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2

    last_out = {}                  # --dump-outputs: the results of the latest step

    def step(batch):
        opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.float16, enabled=amp):
            if ns is None:
                lidar = ts.SparseTensor(batch["feats"], batch["coords"], 1)
                out = net({"lidar": lidar, "targets": batch["labels"]})
            else:
                out = net(ns.batch_dict(batch, dev))[0]
        loss = out["loss"]
        if args.dump_outputs:
            last_out.clear()
            last_out.update(out)
        scaler.scale(loss).backward()
        scaler.unscale_(opt)
        torch.nn.utils.clip_grad_norm_(model.parameters(), 10.0)
        scaler.step(opt)
        scaler.update()
        return loss

    copy_stream = torch.cuda.Stream(device=dev)
    loss_host = [torch.zeros(1, dtype=torch.float32).pin_memory() for _ in range(2)]

    def upload(i):
        """Host -> device copy of step i's inputs from pinned memory on the copy stream (so that it runs under the
        previous step's kernels, as a prefetching loader with pin_memory does) + the event the step waits on."""
        with torch.cuda.stream(copy_stream):
            batch = {k: v.to(dev, non_blocking=True) for k, v in pool[i % len(pool)].items()}
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return batch, ev

    def run(n_steps, from_host):
        """Returns (ms_total over the timed steps [device events, max over ranks], last loss value).
        from_host: every step's inputs are copied from pinned host memory and every step's loss is copied back to
        the host INSIDE the timed region; the loss of step i is read by the host while step i + 1 is queued (an
        asynchronous copy into pinned memory + an event), so the host never drains the device mid-run."""
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        main_stream = torch.cuda.current_stream(dev)
        last, nxt, read_ev = None, None, [None, None]
        ev0.record()
        if from_host:
            nxt = upload(0)
        for i in range(n_steps):
            flush_buf.zero_()                              # L2 flush between iterations
            if from_host:
                batch, ready = nxt
                main_stream.wait_event(ready)
                for t in batch.values():
                    t.record_stream(main_stream)
                if i + 1 < n_steps:
                    nxt = upload(i + 1)
            else:
                batch = resident[i % len(resident)]
            loss = step(batch)
            if from_host:
                loss_host[i % 2].copy_(loss.detach().float().reshape(1), non_blocking=True)   # D2H of the step's result
                read_ev[i % 2] = torch.cuda.Event()
                read_ev[i % 2].record(main_stream)
                if i > 0:
                    read_ev[(i - 1) % 2].synchronize()
                    last = float(loss_host[(i - 1) % 2][0])
        if from_host and n_steps > 0:
            read_ev[(n_steps - 1) % 2].synchronize()
            last = float(loss_host[(n_steps - 1) % 2][0])
        ev1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        return D.max_over_ranks(ev0.elapsed_time(ev1), dev), last

    # every distinct batch of the pool is seen three times before timing: buffer sizes differ per batch (step tables,
    # kernel maps: up to 160 MB each) and the caching allocator only stops calling cudaMalloc after that
    warm = max(args.warmup, 3 * len(pool), 3)
    run(warm, False)

    # ---- timed region 1: device-resident inputs (this is `value`)
    if ours:
        B.STATS["launches"] = 0
    sampler = clocks_sampler() if rank == 0 else None
    ms_dev, _ = run(args.steps, False)
    launches = B.STATS["launches"] if ours else None
    clocks = clocks_summary(sampler) if rank == 0 else None

    # ---- the same steps again with every conv launch bracketed by CUDA events (roofline numbers only:
    # the event pairs cost a few % of throughput, so they stay out of `value`)
    conv, ms_prof = {}, None
    if ours:
        prof = ConvProfiler(n_events=args.steps * 460)
        B.PROFILER = prof
        ms_prof, _ = run(args.steps, False)
        B.PROFILER = None
        conv = prof.summarise()

    # ---- timed region 2: end to end from pinned host buffers
    run(max(2, 2 * len(pool)), True)          # the copy stream has its own allocator pool: let it see every batch size
    ms_e2e, last_loss = run(args.steps, True)
    dumped = None
    if args.dump_outputs:          # every rank takes the step (DDP all-reduces its gradients), rank 0 writes it
        model.load_state_dict(start_state[0])
        opt.load_state_dict(start_state[1])
        scaler = torch.amp.GradScaler("cuda", enabled=amp)
        scale = scaler.get_scale()
        torch.manual_seed(0)
        step(resident[(args.steps - 1) % len(resident)])
        torch.cuda.synchronize()
        if rank == 0:
            dumped = {"dir": args.dump_outputs, "shapes": dump_outputs(args.dump_outputs, last_out, model),
                      "optimizer_step_applied": not amp or scaler.get_scale() >= scale}

    value = D.whole_job_rate(args.batch * args.steps, world, ms_dev)
    e2e = D.whole_job_rate(args.batch * args.steps, world, ms_e2e)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk = peaks()
    # The dominant kernel: forward and input-gradient are the SAME kernel (gather_gemm_tc3_kernel,
    # different maps / weight transposes), the weight gradient is a second kernel (wgrad_tc_kernel).
    roof = None
    if conv:
        fams = {"conv gather-GEMM (fwd+dgrad), gather_gemm_tc3_kernel": ("fwd", "dgrad"),
                "conv wgrad, wgrad_tc_kernel": ("wgrad",)}
        tot = {name: sum(conv[k]["ms"] for k in ks if k in conv) for name, ks in fams.items()}
        name = max(tot, key=tot.get)
        ks = [k for k in fams[name] if k in conv]
        fam_ms = sum(conv[k]["ms"] for k in ks)
        fam_fl = sum(conv[k]["gflop"] for k in ks)
        achieved = (fam_fl / 1e3) / (fam_ms / 1e3)
        peak = pk["tflops_sustained"] if amp else None
        roof = {"kernel": name, "bound": "tensor", "achieved": achieved, "peak": peak,
                "unit": "TFLOP/s", "frac": (achieved / peak) if peak else None,
                "peak_source": pk["source"] + " (sustained bf16 cuBLAS, MEASURED_PEAKS.json)" if amp else
                "fp32 runs on the CUDA-core kernels (1e-5 bar rules out tf32); no tensor peak applies",
                "traffic": 138.4e6, "traffic_detail": TRAFFIC.get(args.config), "launches_timed": sum(conv[k]["launches"] for k in ks),
                "share_of_step": fam_ms / ms_prof,
                "per_family": {k: {kk: round(vv, 4) for kk, vv in v.items()} for k, v in conv.items()},
                "note": "achieved = useful FLOPs 2*M*Cin*Cout (M = kernel-map pairs) / CUDA-event time, "
                        "summed over every launch in the timed region; alg_gbs = algorithmic bytes "
                        "(e*Cin*M + e*Cout*N + 8*M + e*K*Cin*Cout) / the same time; traffic = ncu "
                        "dram__bytes_read+write (bytes) of one representative launch of the dominant kernel "
                        "(L0 96->96 at 4 scans, algorithmic 157.0e6 bytes); other layers in traffic_detail"}

    cpu_info = None
    if world == 1 and ours and not args.no_cpu_baseline:
        try:
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--config",
                                  args.config, "--steps", "1", "--warmup", "0", "--cpu-budget-s",
                                  str(args.cpu_budget_s or 25.0)], capture_output=True, text=True,
                                 timeout=600)
            cpu_info = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])["cpu_baseline"]
        except Exception as exc:                               # never lose the GPU line
            cpu_info = {"value": None, "unit": "scans/s", "cores": os.cpu_count(), "kind": "reference",
                        "sample": f"failed: {exc}"}
    ref_cuda = ref_cuda_child(args) if (world == 1 and ours and not args.no_ref_cuda) else None
    cfg1 = None
    if world == 1 and ours and not args.no_config1:
        try:
            cfg1 = config1_run(dev)
        except Exception as exc:
            cfg1 = {"error": f"{type(exc).__name__}: {str(exc)[:200]}"}

    line = {"metric": metric, "value": value, "unit": "scans/s", "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f16" if amp else "f32", "data": "synthetic",
            "config": {"workload": workload, "name": args.config, "model_src": args.model_src,
                       "scans_per_gpu_per_step": args.batch, "voxels_per_scan": int(vox_per_scan),
                       "amp": amp, "sync_bn": bool(args.sync_bn and world > 1),
                       "parallelism": f"dp{world}", "sm_reserve": reserve, "ddp_bucket_mb": args.bucket_mb,
                       "l2": "256 MiB flush write before every step",
                       "peaks": pk},
            "clocks": clocks,
            "e2e": {"value": e2e, "unit": "scans/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / args.steps, "last_loss": last_loss},
            "gpu_launches": launches,
            "roofline": roof, "cpu_baseline": cpu_info}
    if not ours:
        line["impl"] = args.impl
        line["config"]["backend"] = "reference torchsparse 1.4.0 CUDA backend recompiled for sm_100a (oracle/_ref)"
    else:
        line["ref_cuda"] = ref_cuda
        line["config1"] = cfg1
    if dumped is not None:
        line["dumped_outputs"] = dumped
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ncu `--set full` DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) of one representative launch of
# the dominant family, filled from profiles/ (see profiles/README.md for the capture commands)
_TC4_TRAFFIC = {"unit": "bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum)",
                "gather_gemm_tc4_kernel, L0 96->96, 4 scans (381 k rows, 1.77 M pairs)":
                    {"dram_bytes": 138.4e6, "algorithmic_bytes": 157.0e6, "us": 106.8, "tensor_pipe_pct": 25.5},
                "gather_gemm_tc4_kernel, L3 256->256, 4 scans (39.8 k rows, 328 k pairs)":
                    {"dram_bytes": 26.0e6, "algorithmic_bytes": 47.5e6, "us": 103.1, "tensor_pipe_pct": 45.5},
                "wgrad_tc_kernel, L0 96->96, 4 scans": {"dram_bytes": 420.5e6, "algorithmic_bytes": 160.0e6, "us": 156.9,
                                                        "tensor_pipe_pct": 14.2},
                "source": "profiles/r2_ncu_conv_full.txt"}
TRAFFIC: dict = {c: _TC4_TRAFFIC for c in CONFIGS}


if __name__ == "__main__":
    main()
