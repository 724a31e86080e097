"""Large-graph measurements of the 16-bit inference path (N up to 4096), written as one JSON document.

  python tools/large_graph_bench.py --out large_graphs.json

Measures, on cuda:0, with the card's name and power limit read in the same run:
  * fp16 ms per pair for two embeds plus the fused head (Siamese_Node_Exp.loss_and_accuracy) from inputs resident on
    the device, 4 blocks of depth 3, N in {1024, 2048, 3072, 4096}, C in {32, 64}; TFLOP/s from oracle.flops_per_pair;
  * the same step in fp32 mode (CUDA cores, every (B,C,N,N) intermediate kept) at N = 2048, C = 32;
  * the device linear assignment (fgnn_lap_fwd) at N = 4096, ms per graph;
  * the Regular generator (fgnn_generate_pairs_u8, edge_density 0.2 as in default_config.yaml) at N = 2048 and 4096.
Every timed shape is run once before its window; windows are timed with CUDA events and last at least --min-window
seconds (a single call longer than that is one window).  The inputs of the embed timings (2 x 134 MB fp32 features at
N = 4096) are smaller than the L2 but every embed streams gigabytes of 16-bit planes, so the cache is not what is timed.
"""
import argparse
import json
import os
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
    """Warm-up call, then windows of repeated calls between CUDA events until one lasts >= min_window s: ms per call."""
    fn()
    torch.cuda.synchronize()
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
            return {"ms": ms / reps, "reps": reps, "window_s": ms / 1e3}
        reps = max(reps + 1, int(reps * 1.2e3 * min_window / max(ms, 1e-3)) + 1)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True, help="JSON file to write")
    ap.add_argument("--sizes", default="1024,2048,3072,4096")
    ap.add_argument("--widths", default="32,64")
    ap.add_argument("--min-window", type=float, default=1.0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("large_graph_bench.py measures the GPU: no CUDA device")

    import graph_neural_net_b200 as pkg
    from graph_neural_net_b200 import _ops
    from graph_neural_net_b200.loaders.data_generator import adjacency_batch_to_tensor_representation
    from graph_neural_net_b200.toolbox.metrics import linear_assignment
    from oracle import fgnn_oracle as O

    dev = torch.device("cuda:0")
    res = {"card": card(), "torch": torch.__version__, "time": time.strftime("%Y-%m-%dT%H:%M:%S"),
           "model": {"num_blocks": 4, "depth_of_mlp": 3}, "embed_pair": [], "lap": None, "regular_generator": []}

    def model_for(c, prec):
        gen = torch.Generator().manual_seed(c)
        sd = O.xavier_state_dict(2, c, 4, 3, gen)
        node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=4,
                        in_features=c, out_features=c, depth_of_mlp=3)
        m = pkg.models.Siamese_Node_Exp(2, node_emb)
        m.load_state_dict(sd)
        return m.to(dev).set_precision(prec)

    def pair_inputs(n):
        a1, a2 = _ops.generate_pairs(0, 1, n, 0.2, 0.1, 1234, None, dev)     # ErdosRenyi, p = 0.2
        return adjacency_batch_to_tensor_representation(a1), adjacency_batch_to_tensor_representation(a2)

    runs = [(n, c, "fp16") for c in [int(v) for v in args.widths.split(",")] for n in [int(v) for v in args.sizes.split(",")]]
    runs.append((2048, 32, "fp32"))
    for n, c, prec in runs:
        model = model_for(c, prec)
        x1, x2 = pair_inputs(n)
        step = lambda: model.loss_and_accuracy({"input": x1}, {"input": x2})
        t = timed(step, args.min_window)
        flop = O.flops_per_pair(n, c)
        row = {"n": n, "c": c, "precision": prec, "ms_per_pair": t["ms"], "tflops": flop / (t["ms"] * 1e-3) / 1e12,
               "flop_per_pair": flop, "reps": t["reps"], "window_s": t["window_s"]}
        print(json.dumps(row), flush=True)
        res["embed_pair"].append(row)
        del model, x1, x2
        torch.cuda.empty_cache()

    # linear assignment at N = 4096 on scores with a trained-like diagonal and noise (one CTA per graph)
    gen = torch.Generator().manual_seed(4096)
    scores = (torch.randn((1, 4096, 4096), generator=gen) * 3 + 4 * torch.eye(4096)).to(dev)
    t = timed(lambda: linear_assignment(scores), args.min_window)
    res["lap"] = {"n": 4096, "ms_per_graph": t["ms"], "reps": t["reps"], "window_s": t["window_s"]}
    print(json.dumps(res["lap"]), flush=True)

    # Regular generator (one graph, edge_density 0.2): the switch chain is sequential, so one call can exceed the window
    for n in (2048, 4096):
        t = timed(lambda: _ops.generate_pairs(1, 1, n, 0.2, 0.1, 99, None, dev), args.min_window)
        d = int(0.2 * n)
        row = {"n": n, "edge_density": 0.2, "degree": d, "edges": n * d // 2, "ms_per_graph": t["ms"], "reps": t["reps"],
               "window_s": t["window_s"]}
        print(json.dumps(row), flush=True)
        res["regular_generator"].append(row)

    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
