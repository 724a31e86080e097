#!/usr/bin/env python
"""bench.py -- throughput of the 2-FGNN siamese forward (BASELINE.json metric) on N B200s.

    python bench.py --gpus 1 --steps 5 --warmup 3            # this implementation
    python bench.py --gpus 1 --steps 5 --warmup 3 --dump-outputs DIR   # ... and write the last step's outputs as .npy
    python bench.py --impl reference --steps 3 --warmup 1    # CPU reference arm (oracle port)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload = BASELINE.json configs[2] (the configuration the metric is quoted on): siamese 2-FGNN,
embedding width 64, 4 blocks, depth-3 MLPs, regular graphs n=500 (d=100), ER noise 0.1, 64 pairs
per GPU, 16-bit forward (fp16 operands by default: the 16-bit mode that meets the 2e-2 tolerance).  One step = one siamese forward over the batch: both embedders, the
E1^T E2 scores, and the fused row-softmax CE / argmax head.  Synthetic data, random-init weights.

Prints ONE JSON line (rank 0).  `value` = pairs/s with inputs resident in HBM; `e2e` = the same
through the public Python API from pinned host buffers (H2D of the step's inputs and D2H of the
loss/accuracy inside the timed region).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = {
    # name: (n, width, blocks, depth, pairs per GPU, regular degree or None (ER p=0.2))
    "cfg3_regular_n500_c64_b64_fwd": dict(n=500, c=64, blocks=4, depth=3, pairs=64, regular=True),
    "cfg2_er_n200_c32_b128_fwd": dict(n=200, c=32, blocks=4, depth=3, pairs=128, regular=False),
    "cfg1_er_n50_c32_b32_fwd": dict(n=50, c=32, blocks=4, depth=3, pairs=32, regular=False),
}
DEFAULT_WORKLOAD = "cfg3_regular_n500_c64_b64_fwd"
METRIC = "graph-pairs/sec 2-FGNN siamese fwd at n=500"
DUMP_LIMIT_BYTES = 64 * 10**6


def dump_outputs(out_dir, arrays, seed=0):
    """Write each array as out_dir/<name>.npy: float64 stays float64, everything else is stored as float32.  Arrays
    are indexed by pair along their first axis (0-d arrays are scalars).  When all of them together exceed 64 MB,
    every array keeps the same fixed, seeded sample of pairs, whose indices are written as pair_index.npy."""
    import numpy as np
    host = {k: v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v) for k, v in arrays.items()}
    host = {k: v if v.dtype == np.float64 else v.astype(np.float32) for k, v in host.items()}
    budget = DUMP_LIMIT_BYTES - 4096 * (len(host) + 1)        # room for the .npy headers, pair_index.npy's included
    if sum(v.nbytes for v in host.values()) > budget:
        pairs = max(v.shape[0] for v in host.values() if v.ndim)
        per_pair = sum(v.nbytes // v.shape[0] for v in host.values() if v.ndim) + 8      # + its float64 pair_index entry
        scalars = sum(v.nbytes for v in host.values() if not v.ndim)
        keep = np.sort(np.random.default_rng(seed).choice(pairs, (budget - scalars) // per_pair, replace=False))
        host = {k: v[keep] if v.ndim else v for k, v in host.items()}
        host["pair_index"] = keep.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in host.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(burst=p.get("bf16_tflops", 1590.0), sustained=p.get("bf16_tflops_sustained", 1400.0),
                    hbm=p.get("hbm_gbs", 6650.0), src="measured")
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, src="fallback")


def make_inputs(cfg, pairs, seed):
    """(pairs,2,n,n) fp32 host tensors of both sides.  With a GPU: the reference's generators drawn on the device
    (fgnn_generate_pairs_u8: "Regular" d = int(0.2 n) random regular graphs by the switch chain / "ErdosRenyi" p = 0.2, then
    noise_erdos_renyi(0.1), loaders/data_generator.py:39-87) and expanded by fgnn_features_from_adjacency_u8; without one
    (this container) the oracle's host-side stand-in."""
    if torch.cuda.is_available():
        from graph_neural_net_b200.loaders.data_generator import generate_pairs_on_device, adjacency_batch_to_tensor_representation
        a1, a2 = generate_pairs_on_device("Regular" if cfg["regular"] else "ErdosRenyi", pairs, cfg["n"], 0.2, 0.1, seed=seed)
        x1 = adjacency_batch_to_tensor_representation(a1).cpu()
        x2 = adjacency_batch_to_tensor_representation(a2).cpu()
        del a1, a2
        torch.cuda.empty_cache()
        return x1, x2
    from oracle import fgnn_oracle as O
    gen = torch.Generator().manual_seed(seed)
    n = cfg["n"]
    deg = int(0.2 * n) if cfg["regular"] else None
    x1 = torch.empty((pairs, 2, n, n), dtype=torch.float32)
    x2 = torch.empty((pairs, 2, n, n), dtype=torch.float32)
    for i in range(pairs):
        a, b = O.synthetic_pair(n, 0.2, 0.1, gen, regular_degree=deg)
        x1[i], x2[i] = a, b
    return x1, x2


def make_state_dict(cfg, seed=3787):
    from oracle import fgnn_oracle as O
    gen = torch.Generator().manual_seed(seed)
    return O.xavier_state_dict(2, cfg["c"], cfg["blocks"], cfg["depth"], gen)


class ClockSampler(threading.Thread):
    """SM clock, power and clock-event (throttle) reasons sampled WHILE the timed regions run: NVML polled every 10 ms
    in-process (nvidia_ml_py), or nvidia-smi every 200 ms when NVML cannot be loaded.  A default run's timed region is
    ~150 ms, so the sampler stays on over both timed regions (device-resident and end-to-end)."""

    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = threading.Event()
        self.rows = []            # (sm_mhz, sm_max_mhz, power_w, reason bit mask)
        self.source = None

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            if not uuid.startswith("GPU-"):
                uuid = "GPU-" + uuid
            return pynvml, pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
        except Exception:
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.index)

    def run(self):
        try:
            nv, h = self._nvml_handle()
            smax = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.source = "nvml, 10 ms"
            while not self.stop_flag.is_set():
                try:
                    get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
                    self.rows.append((float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), smax,
                                      nv.nvmlDeviceGetPowerUsage(h) / 1000.0, int(get_reasons(h))))
                except Exception:
                    pass
                self.stop_flag.wait(0.01)
            return
        except Exception:
            pass
        self.source = "nvidia-smi, 200 ms"
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                parts = [p.strip() for p in out.stdout.strip().split(",")]
                if len(parts) >= 7:
                    mask = sum(bit for k, (_, bit) in enumerate(self.REASONS) if parts[3 + k].lower().startswith("active"))
                    self.rows.append((float(parts[0]), float(parts[1]), float(parts[2]), mask))
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(r[0] for r in self.rows)
        reasons = [nm for nm, bit in self.REASONS if any(r[3] & bit for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": self.rows[0][1],
                "power_w_max": max(r[2] for r in self.rows), "samples": len(self.rows), "reasons": reasons,
                "source": self.source, "over": "both timed regions (device-resident and end-to-end)"}


def er_pairs_on_device(pairs, n, p, noise, dev, seed):
    """Erdos-Renyi pairs of the reference's generator (loaders/data_generator.py:39-44, 79-87:
    W_noise = W (1 - N1) + (1 - W) N2, N1 ~ ER(noise), N2 ~ ER(p noise / (1 - p))) drawn with torch on the GPU
    (distributional stand-in used by the secondary lines only) -> two (pairs, 2, n, n) fp32 feature tensors."""
    g = torch.Generator(device=dev).manual_seed(seed)

    def er(prob):
        u = torch.rand((pairs, n, n), device=dev, generator=g)
        a = torch.triu((u < prob).float(), 1)
        return a + a.transpose(1, 2)

    W = er(p)
    Wn = W * (1 - er(noise)) + (1 - W) * er(p * noise / (1 - p))

    def feats(A):
        return torch.stack((A, torch.diag_embed(A.sum(2))), dim=1).contiguous()
    return feats(W), feats(Wn)


def _time_steps(fn, steps, warmup, dev, world):
    import torch.distributed as dist
    for _ in range(warmup):
        fn()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = fn()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms, out


def run_secondaries(pkg, dev, rank, world, precision):
    """Secondary lines for the other BASELINE.json configs (short runs, same timing rules: warm-up >= 3, CUDA events,
    max over ranks).  N = 1: cfg1 / cfg2 forward, cfg2 training step, cfg4 ragged forward and training step.
    N > 1: the cfg5 data-parallel training step with its flat all-reduce, and the fixed-512-pair strong-scaling point."""
    import numpy as np
    import torch.distributed as dist
    from oracle import fgnn_oracle as O
    from graph_neural_net_b200 import _ops
    from graph_neural_net_b200.maskedtensors import maskedtensor as mt
    from graph_neural_net_b200.toolbox.losses import triplet_loss
    from graph_neural_net_b200.training import train_step_flat, FlatAdam
    prec = precision if precision != "fp32" else "fp16"
    dt = {"fp16": "f16", "bf16": "bf16"}[prec]
    out = {}

    def build(c, blocks=4, depth=3, **extra):
        node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=blocks,
                        in_features=c, out_features=c, depth_of_mlp=depth, **extra)
        model = pkg.models.Siamese_Node_Exp(2, node_emb)
        model.load_state_dict(O.xavier_state_dict(2, c, blocks, depth, torch.Generator().manual_seed(3787)))
        return model.to(dev)

    def fwd_line(model, x1, x2, p, flops, steps=5):
        model.set_precision(p)
        loss_fn = triplet_loss()

        def step():
            with torch.no_grad():
                return loss_fn(model(x1, x2))
        ms, _ = _time_steps(step, steps, 3, dev, world)
        pairs = (x1["input"].shape[0] if not isinstance(x1["input"], mt.MaskedTensor) else len(x1["input"])) * world
        return {"value": pairs * steps / (ms / 1e3), "unit": "pairs/s", "ms_per_step": ms / steps, "dtype": {"fp32": "f32"}.get(p, dt),
                "tflops": flops * world * steps / (ms / 1e3) / 1e12}

    def train_line(model, x1, x2, flops_fwd, steps=4):
        model.set_precision(prec)
        opt = FlatAdam(model.parameters(), lr=model.lr)
        ms, res = _time_steps(lambda: train_step_flat(model, opt, x1, x2), steps, 3, dev, world)
        pairs = (x1["input"].shape[0] if not isinstance(x1["input"], mt.MaskedTensor) else len(x1["input"])) * world
        return {"value": pairs * steps / (ms / 1e3), "unit": "pairs/s", "ms_per_step": ms / steps, "dtype": dt,
                "tflops": 3 * flops_fwd * world * steps / (ms / 1e3) / 1e12, "final_loss": res[0],
                "what": "fwd + tcgen05 bwd + one flat all-reduce + fused flat Adam (fgnn_embed_fwd_train / fgnn_embed_bwd)"}

    if world == 1:
        m32 = build(32)
        a, b = er_pairs_on_device(32, 50, 0.2, 0.1, dev, 1)
        f1 = O.flops_per_pair(50, 32) * 32
        out["cfg1_er_n50_c32_b32_fwd"] = {"fp32": fwd_line(m32, {"input": a}, {"input": b}, "fp32", f1),
                                          prec: fwd_line(m32, {"input": a}, {"input": b}, prec, f1)}
        a, b = er_pairs_on_device(128, 200, 0.2, 0.1, dev, 2)
        f2 = O.flops_per_pair(200, 32) * 128
        out["cfg2_er_n200_c32_b128_fwd"] = fwd_line(m32, {"input": a}, {"input": b}, prec, f2)
        out["cfg2_er_n200_c32_b128_train"] = train_line(build(32), {"input": a}, {"input": b}, f2)
        del a, b
        # cfg4: ragged MaskedTensor batch, n_b ~ UniformInt[50, 1000] (numpy default_rng(3787)), in-kernel masking
        rng = np.random.default_rng(3787)
        sizes = [int(v) for v in rng.integers(50, 1001, size=16)]
        g1, g2 = [], []
        for i, nb in enumerate(sizes):
            a, b = er_pairs_on_device(1, nb, 0.2, 0.1, dev, 100 + i)
            g1.append(a[0].cpu())
            g2.append(b[0].cpu())
        f4 = sum(O.flops_per_pair(nb, 32) for nb in sizes)
        mr = build(32, constant_n_vertices=False)
        x1 = {"input": mt.from_list(g1, dims=(1, 2)).to(dev)}
        x2 = {"input": mt.from_list(g2, dims=(1, 2)).to(dev)}
        line = fwd_line(mr, x1, x2, prec, f4, steps=3)
        line["sizes"] = sizes
        line["flops"] = "sum over graphs of the SURVEY 8(d) formula at each n_b (never at Nmax)"
        out["cfg4_ragged_n50_1000_c32_b16_fwd"] = line
        k = 4
        x1 = {"input": mt.from_list(g1[:k], dims=(1, 2)).to(dev)}
        x2 = {"input": mt.from_list(g2[:k], dims=(1, 2)).to(dev)}
        tl = train_line(build(32, constant_n_vertices=False), x1, x2, sum(O.flops_per_pair(nb, 32) for nb in sizes[:k]), steps=3)
        tl["sizes"] = sizes[:k]
        out["cfg4_ragged_c32_b4_train"] = tl
        pkg._lib.release_workspaces()
        torch.cuda.empty_cache()
    else:
        # cfg5: data-parallel training step, ER n=100, 128 pairs per GPU (global 128 N), ONE flat all-reduce per step
        a, b = er_pairs_on_device(128, 100, 0.2, 0.1, dev, 50 + rank)
        model = build(32)
        f5 = O.flops_per_pair(100, 32) * 128
        tl = train_line(model, {"input": a}, {"input": b}, f5, steps=5)
        nparam = sum(p.numel() for p in model.parameters())
        buf = torch.zeros(nparam + 4, device=dev)
        ms_ar, _ = _time_steps(lambda: dist.all_reduce(buf), 20, 5, dev, world)
        tl["allreduce_us"] = ms_ar / 20 * 1e3
        tl["allreduce_bytes"] = int(buf.numel() * 4)
        tl["collective"] = "one NCCL all-reduce (sum) of the flat fp32 buffer [all gradients | sum CE, rows, correct, overflow flag]"
        out[f"cfg5_er_n100_c32_dp{world}_train"] = tl
        del a, b
        # strong scaling: a fixed global batch of 512 cfg3 pairs (64-wide, regular-degree-like density) over N GPUs
        per = 512 // world
        m64 = build(64)
        m64.set_precision(prec)
        a, b = er_pairs_on_device(min(per, 64), 500, 0.2, 0.1, dev, 70 + rank)
        reps = max(1, per // a.shape[0])

        def strong():
            with torch.no_grad():
                for _ in range(reps):
                    s = m64({"input": a}, {"input": b})
            return s
        ms, _ = _time_steps(strong, 2, 3, dev, world)
        out["cfg3_strong_512_pairs"] = {"value": 512 * 2 / (ms / 1e3), "unit": "pairs/s", "ms_per_512_pairs": ms / 2,
                                        "pairs_per_gpu": per, "dtype": dt, "inputs": "ER p=0.2 n=500 (same dense shapes as cfg3)"}
    return out


def _unmodified_reference_step(cfg, sd):
    """The UNMODIFIED reference (imported through oracle/refshim.py) as the CPU arm, when its tree is present -- it is
    not on the GPU box, where the oracle port stands in.  Returns step(x1, x2) -> loss, or None."""
    try:
        from oracle import refshim
        if not os.path.isdir(refshim.REFERENCE_ROOT):
            return None
        refshim.install()
        import models as ref_models                        # the reference's own package
        from toolbox.losses import triplet_loss as ref_loss
        arch = {"original_features_num": 2,
                "node_emb": dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=cfg["blocks"],
                                 in_features=cfg["c"], out_features=cfg["c"], depth_of_mlp=cfg["depth"])}
        model = ref_models.get_siamese_model_exp(arch, {"lr": 1e-3, "scheduler_decay": 0.5, "scheduler_step": 3})
        model.load_state_dict(sd)
        model.eval()
        loss_fn = ref_loss()
        return lambda x1, x2: float(loss_fn(model({"input": x1}, {"input": x2})))
    except Exception as e:                                 # noqa: BLE001 - any import problem: fall back to the port
        print(f"[bench] unmodified reference unavailable ({type(e).__name__}: {e}); timing the oracle port", file=sys.stderr)
        return None


def cpu_reference_rate(cfg, steps, warmup, pairs_per_step=1):
    """The reference algorithm on the host cores (fp32 torch CPU, all threads) on a bounded sample: the unmodified
    reference when /root/reference exists (kind "reference"), else its oracle port (kind "port")."""
    from oracle import fgnn_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sd = make_state_dict(cfg)
    x1, x2 = make_inputs(cfg, pairs_per_step, seed=11)
    ref_step = _unmodified_reference_step(cfg, sd)
    kind = "reference" if ref_step is not None else "port"
    times = []
    with torch.no_grad():
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            if ref_step is not None:
                ref_step(x1, x2)
            else:
                float(O.triplet_loss(O.siamese_forward(x1, x2, sd)))
            dt = time.perf_counter() - t0
            if it >= warmup:
                times.append(dt)
    total = sum(times)
    return pairs_per_step * len(times) / total, cores, total / len(times), kind


def run_reference(args, cfg, rank, world):
    if rank != 0:
        return
    rate, cores, sec, kind = cpu_reference_rate(cfg, args.steps, args.warmup)
    what = "unmodified reference imported through oracle/refshim.py" if kind == "reference" else "oracle port (no reference tree on this box)"
    sample = f"1 pair per step ({args.steps} timed steps, {args.warmup} warm-up) of the same workload, {what}, fp32 torch CPU"
    line = {"impl": "reference", "metric": METRIC, "value": rate, "unit": "pairs/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "n": cfg["n"], "width": cfg["c"], "blocks": cfg["blocks"],
                       "pairs_per_step": 1},
            "cpu_baseline": {"value": rate, "unit": "pairs/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": rate, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="fp16", choices=["bf16", "fp16", "fp32"],
                    help="fp16 (default) is the 16-bit mode that meets the north_star 2e-2 embedding tolerance against the "
                         "reference at this shape (tests/test_gpu_tc.py); bf16 runs the same tcgen05 kind::f16 kernels")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary lines (cfg1 / cfg2 / cfg4 / cfg5)")
    ap.add_argument("--pairs", type=int, default=0, help="override pairs per GPU (profiling runs only)")
    ap.add_argument("--train", action="store_true",
                    help="time the data-parallel TRAINING step (fwd + bwd + flat all-reduce + Adam) in --precision "
                         "instead of the forward; secondary line for configs[1]/[4], not the headline")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed on rank 0 as DIR/<name>.npy "
                         "(forward: per-pair CE sums, correct rows and both embedding batches; --train: loss, correct, "
                         "rows); inputs and weights are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of this implementation's timed step (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    cfg = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, cfg, rank, world)
        return

    import torch.distributed as dist
    import graph_neural_net_b200 as pkg
    from graph_neural_net_b200.toolbox.losses import triplet_loss
    from graph_neural_net_b200 import _ops

    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=ours) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib = pkg.get_lib()
    peaks = load_peaks()

    pairs = args.pairs if args.pairs > 0 else cfg["pairs"]
    node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=cfg["blocks"],
                    in_features=cfg["c"], out_features=cfg["c"], depth_of_mlp=cfg["depth"])
    model = pkg.models.Siamese_Node_Exp(2, node_emb)
    model.load_state_dict(make_state_dict(cfg))
    model = model.to(dev).set_precision(args.precision)
    loss_fn = triplet_loss()

    if args.train:
        from graph_neural_net_b200.training import train_step_flat as train_step, FlatAdam
        opt = FlatAdam(model.parameters(), lr=model.lr)
        x1_h, x2_h = make_inputs(cfg, pairs, seed=100 + rank)
        b1, b2 = {"input": x1_h.to(dev)}, {"input": x2_h.to(dev)}
        for _ in range(args.warmup):
            train_step(model, opt, b1, b2)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            loss, ok, rows = train_step(model, opt, b1, b2)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
            dist.destroy_process_group()
        if rank == 0 and args.dump_outputs:
            dump_outputs(args.dump_outputs, {"loss": float(loss), "correct": float(ok), "rows": float(rows)})
        if rank == 0:
            print(json.dumps({"metric": "graph-pairs/sec 2-FGNN siamese training step (fwd+bwd+allreduce+Adam)",
                              "value": pairs * world * args.steps / (ms / 1e3), "unit": "pairs/s", "n_gpus": world,
                              "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
                              "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                              "dtype": {"fp32": "f32", "fp16": "f16", "bf16": "bf16"}[args.precision],
                              "data": "synthetic", "final_loss": loss, "gpu_launches": int(lib.fgnn_launch_count()),
                              "config": {"workload": args.workload + "+train", "n": cfg["n"], "width": cfg["c"],
                                         "pairs_per_gpu": pairs, "collective": "one flat fp32 all-reduce per step"}}),
                  flush=True)
        return

    x1_h, x2_h = make_inputs(cfg, pairs, seed=100 + rank)
    x1_h, x2_h = x1_h.pin_memory(), x2_h.pin_memory()
    x1_d, x2_d = x1_h.to(dev), x2_h.to(dev)
    res_h = torch.empty(2, dtype=torch.float32).pin_memory()

    def head(e1, e2):
        # 16-bit modes: fused tensor-core head (fgnn_head_fwd: E1^T E2 + row softmax CE + argmax, no (B,N,N) scores in HBM)
        if args.precision == "fp32":
            scores = _ops.ScoresFunction.apply(e1, e2, None)
            return _ops.CrossEntropyIdentityFunction.apply(scores, None)
        return _ops.head_fused(e1, e2, None, args.precision)[:2]

    def step_resident():
        e1 = model.embed({"input": x1_d})
        e2 = model.embed({"input": x2_d})
        return (*head(e1, e2), e1, e2)

    copy_stream = torch.cuda.Stream(device=dev)
    x2_ready = torch.cuda.Event()
    x2_free = torch.cuda.Event()
    x2_free.record()
    # e2e input pipeline (what a loader does): both H2D copies of a step run on a side stream.  x2 is copied under the
    # first embedder pass of the same step; x1 of the NEXT step is copied under the second pass into the other of two
    # device buffers.  The first step of a run copies its own x1 on the main stream (exposed), so every step's inputs
    # are copied from pinned host memory inside the timed region.
    x1_bufs = [x1_d, torch.empty_like(x1_d)]
    x1_ready = [torch.cuda.Event(), torch.cuda.Event()]
    x1_free = [torch.cuda.Event(), torch.cuda.Event()]
    for ev in x1_free:
        ev.record()
    pipe = {"k": 0, "primed": False}

    def step_e2e():
        main = torch.cuda.current_stream(dev)
        cur = pipe["k"] & 1
        nxt = cur ^ 1
        if not pipe["primed"]:
            x1_bufs[cur].copy_(x1_h, non_blocking=True)
            pipe["primed"] = True
        else:
            main.wait_event(x1_ready[cur])
        copy_stream.wait_event(x2_free)              # previous step's reads of x2_d are done
        with torch.cuda.stream(copy_stream):
            x2_d.copy_(x2_h, non_blocking=True)
            x2_ready.record(copy_stream)
            copy_stream.wait_event(x1_free[nxt])     # the step before last has finished reading that buffer
            x1_bufs[nxt].copy_(x1_h, non_blocking=True)
            x1_ready[nxt].record(copy_stream)
        e1 = model.embed({"input": x1_bufs[cur]})
        x1_free[cur].record(main)
        main.wait_event(x2_ready)
        e2 = model.embed({"input": x2_d})
        x2_free.record(main)
        ce, correct = head(e1, e2)
        res = torch.stack((ce.sum() / (pairs * cfg["n"]), correct.sum().float()))
        res_h.copy_(res, non_blocking=False)       # device -> host read of loss and #correct
        pipe["k"] += 1
        return res_h

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps):
        """(ms over `steps` calls of fn, what the last call returned); no step's result is held across the next step."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps - 1):
            fn()
        last = fn()
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, last

    with torch.no_grad():
        for _ in range(args.warmup):
            step_resident()
        torch.cuda.synchronize(dev)
        # ---- device-resident timed region (with per-kernel-class events and clock sampling) ----
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        lib.fgnn_profile_reset()
        lib.fgnn_profile_enable(1)
        lib.fgnn_reset_launch_count()
        ms, last = timed(step_resident, args.steps)
        launches = int(lib.fgnn_launch_count())
        lib.fgnn_profile_enable(0)
        outputs = None
        if args.dump_outputs:
            outputs = {k: t.cpu() for k, t in zip(("ce_sum", "correct", "emb1", "emb2"), last)}
        del last
        import ctypes as C
        kinds = {}
        for kind, name in ((0, "tc_mlp_kernel"), (1, "tc_matmul_kernel"), (2, "plane_stats16_kernel")):
            tot, cnt = C.c_double(0), C.c_int64(0)
            lib.fgnn_profile_read(kind, C.byref(tot), C.byref(cnt))
            kinds[name] = (tot.value, cnt.value)
        # ---- end-to-end timed region ----
        for _ in range(2):
            step_e2e()
        torch.cuda.synchronize(dev)
        pipe["primed"] = False                       # the timed run starts with an exposed copy of its own first input
        ms_e2e, _ = timed(step_e2e, args.steps)
        if rank == 0:
            sampler.stop_flag.set()
            sampler.join(timeout=3)
        # ---- the same through Siamese_Node_Exp.forward, whose result is the (B,N,N) scores the reference's callers get:
        # exposed (un-pipelined) H2D of both inputs, both embedders, tensor-core E1^T E2, D2H of the scores
        scores_h = torch.empty((pairs, cfg["n"], cfg["n"]), dtype=torch.float32).pin_memory()

        def step_e2e_scores():
            x1_d.copy_(x1_h, non_blocking=True)
            x2_d.copy_(x2_h, non_blocking=True)
            scores_h.copy_(model({"input": x1_d}, {"input": x2_d}), non_blocking=False)

        # ---- the same step fed from uint8 adjacency matrices (SURVEY 8(f) row 2): 1 byte per entry over PCIe instead of 8,
        # input features built on the device; un-pipelined copies
        e2e_adj = None
        if args.precision != "fp32":
            a1_h = (x1_h[:, 0] != 0).to(torch.uint8).pin_memory()
            a2_h = (x2_h[:, 0] != 0).to(torch.uint8).pin_memory()
            a1_d, a2_d = torch.empty_like(a1_h, device=dev), torch.empty_like(a2_h, device=dev)

            def step_e2e_adj():
                a1_d.copy_(a1_h, non_blocking=True)
                a2_d.copy_(a2_h, non_blocking=True)
                loss, ok, _ = model.loss_and_accuracy_from_adjacency(a1_d, a2_d)
                res_h.copy_(torch.stack((loss, ok.float())), non_blocking=False)

            step_e2e_adj()
            ms_adj, _ = timed(step_e2e_adj, args.steps)
            e2e_adj = {"value": pairs * world * args.steps / (ms_adj / 1e3), "unit": "pairs/s",
                       "h2d_bytes_per_step": int(a1_h.numel() * 2), "d2h_bytes_per_step": 8,
                       "what": "model.loss_and_accuracy_from_adjacency(adj1, adj2): uint8 adjacency from pinned host memory, "
                               "features built on the device (fgnn_embed_fwd_adjacency_u8); H2D copies not pipelined"}
        step_e2e_scores()
        k_sc = max(2, args.steps // 4)
        ms_sc, _ = timed(step_e2e_scores, k_sc)
        e2e_scores = {"value": pairs * world * k_sc / (ms_sc / 1e3), "unit": "pairs/s", "steps": k_sc,
                      "d2h_bytes_per_step": int(scores_h.numel() * 4),
                      "what": "model.forward(x1, x2) with the (B,N,N) fp32 scores copied back to pinned host memory; "
                              "H2D copies not pipelined"}

    secondary = None
    if not args.no_secondary and args.workload == DEFAULT_WORKLOAD and args.pairs == 0:
        del x1_d, x2_d, x1_bufs
        pkg._lib.release_workspaces()
        torch.cuda.empty_cache()
        secondary = run_secondaries(pkg, dev, rank, world, args.precision)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)

    from oracle import fgnn_oracle as O
    total_pairs = pairs * world * args.steps
    value = total_pairs / (ms / 1e3)
    e2e_value = total_pairs / (ms_e2e / 1e3)
    flops_pair = O.flops_per_pair(cfg["n"], cfg["c"], cfg["blocks"], cfg["depth"])
    f_conv, f_mm = O.flops_per_graph(cfg["n"], cfg["c"], cfg["blocks"], cfg["depth"])
    graphs_per_step = 2 * pairs
    kind_flops = {"tc_mlp_kernel": f_conv * graphs_per_step * args.steps,
                  "tc_matmul_kernel": f_mm * graphs_per_step * args.steps}
    kernels = {}
    for name, (tot_ms, cnt) in kinds.items():
        entry = {"launches": cnt, "total_ms": tot_ms, "share_of_step": tot_ms / ms if ms else None}
        if name in kind_flops and tot_ms > 0:
            entry["tflops"] = kind_flops[name] / (tot_ms / 1e3) / 1e12
        kernels[name] = entry
    dom = max(("tc_mlp_kernel", "tc_matmul_kernel"), key=lambda k: kinds[k][0])
    roofline = None
    if args.precision != "fp32" and kinds[dom][0] > 0:
        achieved = kind_flops[dom] / (kinds[dom][0] / 1e3) / 1e12
        peak = peaks["sustained"]
        # DRAM traffic of the dominant kernel from the committed ncu --set full capture (bytes per graph per
        # launch, averaged over the kernel's instantiations), scaled to this run's graphs per launch
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath) and cfg["n"] == 500 and cfg["c"] == 64:
            with open(tpath) as f:
                tj = json.load(f)
            if dom in tj:
                graphs_per_launch = graphs_per_step * args.steps * tj[dom]["launches_per_graph_block"] * cfg["blocks"] \
                    / max(kinds[dom][1], 1)
                traffic = tj[dom]["dram_bytes_per_graph_launch"] * graphs_per_launch
        roofline = {"bound": "tensor", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                    "frac": achieved / peak, "traffic": traffic,
                    "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peaks['src']}); kernel timed inside a long step",
                    "flops_per_launch": kind_flops[dom] / max(kinds[dom][1], 1),
                    "avg_launch_ms": kinds[dom][0] / max(kinds[dom][1], 1)}
    line = {
        "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": {"bf16": "bf16", "fp16": "f16", "fp32": "f32"}[args.precision],
        "data": "synthetic (random regular d=100 graphs drawn on the device by the switch chain + Erdos-Renyi noise 0.1; random-init weights)" if cfg["regular"] else "synthetic (Erdos-Renyi p=0.2 + noise 0.1 drawn on the device; random-init weights)",
        "config": {"workload": args.workload, "n": cfg["n"], "width": cfg["c"], "blocks": cfg["blocks"],
                   "depth_of_mlp": cfg["depth"], "pairs_per_gpu": pairs, "global_pairs": pairs * world,
                   "parallelism": f"dp{world} (pairs sharded, no forward collective)",
                   "l2_policy": "inputs (256 MB/step/GPU) and activations (>10 GB/step/GPU) exceed the 126 MB L2"},
        "whole_step_tflops": flops_pair * pairs * world * args.steps / (ms / 1e3) / 1e12,
        "frac_of_bf16_peak_burst": flops_pair * pairs * args.steps / (ms / 1e3) / 1e12 / peaks["burst"],
        "frac_of_bf16_peak_sustained": flops_pair * pairs * args.steps / (ms / 1e3) / 1e12 / peaks["sustained"],
        "gpu_launches": launches,
        "kernels": kernels,
        "roofline": roofline,
        "clocks": sampler.summary(),
        "e2e": {"value": e2e_value, "unit": "pairs/s", "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": int(x1_h.numel() * 4 * 2), "d2h_bytes_per_step": int(res_h.numel() * 4),
                "pipeline": "H2D on a side stream: x2 under this step's first embedder pass, next step's x1 under the "
                            "second (double-buffered); the run's first step copies its own x1 exposed",
                "result": "loss (sum CE / sum n) and #correct rows, 8 bytes: the fused head never writes the (B,N,N) scores; "
                          "the reference API's forward() returns them -- see with_scores",
                "with_scores": e2e_scores, "from_adjacency_u8": e2e_adj},
    }
    if secondary is not None:
        line["secondary"] = secondary
    if world == 1 and not args.no_cpu_baseline:
        rate, cores, sec, kind = cpu_reference_rate(cfg, steps=2, warmup=1)
        line["cpu_baseline"] = {"value": rate, "unit": "pairs/s", "cores": cores, "kind": kind,
                                "sample": f"2 timed + 1 warm-up forwards of 1 pair of the same workload ({sec:.2f} s each), "
                                          + ("unmodified reference via oracle/refshim.py" if kind == "reference" else "oracle port")
                                          + ", fp32 torch CPU"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
