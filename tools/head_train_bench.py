"""Time and memory of the siamese head in training: the fused tensor-core head (fgnn_head_fwd_train + fgnn_head_bwd,
_ops.HeadFunction) against the CUDA-core path (ScoresFunction + CrossEntropyIdentityFunction), as one JSON document.

  python tools/head_train_bench.py --out head_train.json

Measures, on cuda:0, with the card's name and power limit read in the same run:
  * head alone: forward + backward of sum_g ce_sum[g] on resident fp32 embeddings e1 = e2 + noise (requires_grad),
    fp16, at (pairs, C, N) = (32, 32, 50), (128, 32, 200), (64, 64, 500), (16, 64, 1024), (2, 64, 4096): ms per call
    and the peak memory torch allocated above the inputs during one call;
  * whole step: training.train_step_flat with fused_head False and True, fp16, 4 blocks of depth 3, ErdosRenyi
    p = 0.2 pairs drawn on the device, at cfg2 (128 pairs, n = 200, C = 32) and 128 pairs of n = 100, C = 32.
The two arms are alternated for --rounds rounds; each round times a window of repeated calls between CUDA events that
lasts at least --min-window seconds (every training step ends in its own host synchronisation); the medians over the
rounds are reported.  The embeddings (at most 2 x 67 MB) fit the 126 MB L2 at the smaller shapes: those numbers are
warm-cache numbers, as they are inside a training step.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = [v.strip() for v in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def timed(fn, min_window):
    """Windows of repeated calls between CUDA events until one lasts >= min_window s: ms per call."""
    reps = 1
    while True:
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        for _ in range(reps):
            fn()
        stop.record()
        stop.synchronize()
        ms = start.elapsed_time(stop)
        if ms >= 1e3 * min_window:
            return ms / reps
        reps = max(reps + 1, int(reps * 1.2e3 * min_window / max(ms, 1e-3)) + 1)


def alternate(arms, rounds, min_window):
    """{name: fn} -> {name: (median ms, [ms per round])}, arms alternated round by round."""
    times = {k: [] for k in arms}
    for fn in arms.values():                               # warm-up of every arm
        for _ in range(2):
            fn()
    torch.cuda.synchronize()
    for _ in range(rounds):
        for k, fn in arms.items():
            times[k].append(timed(fn, min_window))
    return {k: (statistics.median(v), v) for k, v in times.items()}


def peak_above(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True, help="JSON file to write")
    ap.add_argument("--min-window", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("head_train_bench.py measures the GPU: no CUDA device")

    import graph_neural_net_b200 as pkg
    from graph_neural_net_b200 import _ops
    from graph_neural_net_b200.training import train_step_flat, FlatAdam
    from oracle import fgnn_oracle as O

    dev = torch.device("cuda:0")
    res = {"card": card(), "torch": torch.__version__, "time": time.strftime("%Y-%m-%dT%H:%M:%S"), "precision": "fp16",
           "head": [], "step": []}

    for pairs, c, n in ((32, 32, 50), (128, 32, 200), (64, 64, 500), (16, 64, 1024), (2, 64, 4096)):
        gen = torch.Generator().manual_seed(n)
        e2 = torch.randn(pairs, c, n, generator=gen) * (4.0 / c) ** 0.5
        e1 = (e2 + 0.5 * torch.randn(pairs, c, n, generator=gen) * (4.0 / c) ** 0.5).to(dev).requires_grad_(True)
        e2 = e2.to(dev).requires_grad_(True)

        def fused():
            e1.grad = e2.grad = None
            _ops.HeadFunction.apply(e1, e2, None, "fp16")[0].sum().backward()

        def cuda_core():
            e1.grad = e2.grad = None
            s = _ops.ScoresFunction.apply(e1, e2, None)
            _ops.CrossEntropyIdentityFunction.apply(s, None)[0].sum().backward()

        t = alternate({"fused": fused, "cuda_core": cuda_core}, args.rounds, args.min_window)
        mem = {"fused": peak_above(fused), "cuda_core": peak_above(cuda_core)}
        row = {"pairs": pairs, "c": c, "n": n,
               "fused_ms": t["fused"][0], "cuda_core_ms": t["cuda_core"][0], "speedup": t["cuda_core"][0] / t["fused"][0],
               "fused_ms_rounds": t["fused"][1], "cuda_core_ms_rounds": t["cuda_core"][1],
               "fused_peak_mb": mem["fused"] / 2**20, "cuda_core_peak_mb": mem["cuda_core"] / 2**20}
        print(json.dumps(row), flush=True)
        res["head"].append(row)
        del e1, e2
        torch.cuda.empty_cache()

    for label, pairs, n, c in (("cfg2", 128, 200, 32), ("cfg5 per GPU", 128, 100, 32)):
        gen = torch.Generator().manual_seed(c)
        sd = O.xavier_state_dict(2, c, 4, 3, gen)
        node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=4,
                        in_features=c, out_features=c, depth_of_mlp=3)
        model = pkg.models.Siamese_Node_Exp(2, node_emb)
        model.load_state_dict(sd)
        model = model.to(dev).set_precision("fp16")
        opt = FlatAdam(model.parameters(), lr=model.lr)
        a1, a2 = _ops.generate_pairs(0, pairs, n, 0.2, 0.1, 1234, None, dev)
        b1, b2 = {"input": _ops.features_from_adjacency(a1, None)}, {"input": _ops.features_from_adjacency(a2, None)}
        t = alternate({"default": lambda: train_step_flat(model, opt, b1, b2),
                       "fused_head": lambda: train_step_flat(model, opt, b1, b2, fused_head=True)},
                      args.rounds, args.min_window)
        row = {"label": label, "pairs": pairs, "n": n, "c": c,
               "default_ms": t["default"][0], "fused_head_ms": t["fused_head"][0],
               "saved_fraction": 1.0 - t["fused_head"][0] / t["default"][0],
               "default_ms_rounds": t["default"][1], "fused_head_ms_rounds": t["fused_head"][1]}
        print(json.dumps(row), flush=True)
        res["step"].append(row)
        del model, opt, b1, b2
        torch.cuda.empty_cache()

    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
