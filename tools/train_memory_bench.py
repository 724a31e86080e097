"""Time and memory of the 16-bit training step on its two plans (keep-all / recompute in passes), as one JSON document.

  python tools/train_memory_bench.py --out train_memory.json

Measures, on cuda:0, with the card's name and power limit read in the same run, one training.train_step_flat step
(two embedder calls fgnn_embed_fwd_train + fgnn_embed_bwd, scores, cross-entropy, flat Adam), fp16, 4 blocks of
depth 3, ErdosRenyi p = 0.2 pairs drawn on the device:
  * cfg2 (n = 200, C = 32, 128 pairs) on keep-all and on the recompute plan forced with FGNN_TC_TRAIN_WS_GB=0,
    alternated in windows of the same run: the cost of recomputing;
  * 64 pairs of n = 500, C = 64 (cfg3's architecture and batch), on the plan the default threshold picks;
  * 16 pairs of N = 1024, C = 64, likewise.
For each: ms per step, pairs/s, the plan and workspace bytes of one embedder call, and the peak memory torch allocated
during the timed steps.  Windows are timed with CUDA events and last at least --min-window seconds; every step ends in
the step's own host synchronisation (the loss read-back).
"""
import argparse
import ctypes
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
            return {"ms": ms / reps, "reps": reps, "window_s": ms / 1e3}
        reps = max(reps + 1, int(reps * 1.2e3 * min_window / max(ms, 1e-3)) + 1)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True, help="JSON file to write")
    ap.add_argument("--min-window", type=float, default=2.0)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of keep-all / recompute at cfg2")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("train_memory_bench.py measures the GPU: no CUDA device")
    for v in ("FGNN_TC_TRAIN_WS_GB", "FGNN_TC_WS_GB", "FGNN_TC_CHUNK"):
        os.environ.pop(v, None)

    import graph_neural_net_b200 as pkg
    from graph_neural_net_b200 import _lib as L, _ops
    from graph_neural_net_b200.training import train_step_flat, FlatAdam
    from oracle import fgnn_oracle as O

    dev = torch.device("cuda:0")
    res = {"card": card(), "torch": torch.__version__, "time": time.strftime("%Y-%m-%dT%H:%M:%S"),
           "model": {"num_blocks": 4, "depth_of_mlp": 3, "precision": "fp16"}, "runs": []}

    def setup(n, c, pairs):
        gen = torch.Generator().manual_seed(c)
        sd = O.xavier_state_dict(2, c, 4, 3, gen)
        node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=4,
                        in_features=c, out_features=c, depth_of_mlp=3)
        model = pkg.models.Siamese_Node_Exp(2, node_emb)
        model.load_state_dict(sd)
        model = model.to(dev).set_precision("fp16")
        opt = FlatAdam(model.parameters(), lr=model.lr)
        a1, a2 = _ops.generate_pairs(0, pairs, n, 0.2, 0.1, 1234, None, dev)
        x1, x2 = _ops.features_from_adjacency(a1, None), _ops.features_from_adjacency(a2, None)
        return model, opt, {"input": x1}, {"input": x2}

    def plan_of(model, pairs, n, c):
        """(plan, workspace bytes of one embedder call) as the library picks them now."""
        lib = L.get_lib()
        keep = []
        params = model.node_embedder._embed_params(keep)
        now = lib.fgnn_embed_train_workspace_bytes(ctypes.byref(params), L.PRECISIONS["fp16"], pairs, n)
        saved = os.environ.get("FGNN_TC_TRAIN_WS_GB")
        os.environ["FGNN_TC_TRAIN_WS_GB"] = "1000000"
        keep_all = lib.fgnn_embed_train_workspace_bytes(ctypes.byref(params), L.PRECISIONS["fp16"], pairs, n)
        if saved is None:
            del os.environ["FGNN_TC_TRAIN_WS_GB"]
        else:
            os.environ["FGNN_TC_TRAIN_WS_GB"] = saved
        return ("keep-all" if now == keep_all else "recompute"), now, keep_all

    def measure(label, n, c, pairs, model, opt, b1, b2):
        plan, ws, ws_keep_all = plan_of(model, pairs, n, c)
        step = lambda: train_step_flat(model, opt, b1, b2)
        for _ in range(2):
            step()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        t = timed(step, args.min_window)
        loss = step()[0]
        row = {"label": label, "n": n, "c": c, "pairs": pairs, "plan": plan, "ms_per_step": t["ms"],
               "pairs_per_s": pairs / (t["ms"] * 1e-3), "peak_allocated_gb": torch.cuda.max_memory_allocated() / 1e9,
               "workspace_gb_per_call": ws / 1e9, "keep_all_workspace_gb_per_call": ws_keep_all / 1e9,
               "loss": loss, "reps": t["reps"], "window_s": t["window_s"]}
        print(json.dumps(row), flush=True)
        res["runs"].append(row)
        return row

    # cfg2: keep-all and the forced recompute plan, alternated on the same model and batch
    model, opt, b1, b2 = setup(200, 32, 128)
    cfg2 = {"keep-all": [], "recompute": []}
    for r in range(args.rounds):
        for plan in ("keep-all", "recompute"):
            if plan == "recompute":
                os.environ["FGNN_TC_TRAIN_WS_GB"] = "0"
            else:
                os.environ.pop("FGNN_TC_TRAIN_WS_GB", None)
            cfg2[plan].append(measure(f"cfg2 {plan} round {r}", 200, 32, 128, model, opt, b1, b2)["ms_per_step"])
    os.environ.pop("FGNN_TC_TRAIN_WS_GB", None)
    k, rc = statistics.median(cfg2["keep-all"]), statistics.median(cfg2["recompute"])
    res["cfg2_recompute_overhead"] = {"keep_all_ms_median": k, "recompute_ms_median": rc, "ratio": rc / k}
    print(json.dumps(res["cfg2_recompute_overhead"]), flush=True)
    del model, opt, b1, b2
    torch.cuda.empty_cache()

    # shapes whose keep-all step does not fit one device: the default threshold picks the recompute plan
    for n, c, pairs in ((500, 64, 64), (1024, 64, 16)):
        model, opt, b1, b2 = setup(n, c, pairs)
        measure(f"n{n} c{c} {pairs} pairs", n, c, pairs, model, opt, b1, b2)
        del model, opt, b1, b2
        torch.cuda.empty_cache()

    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
