"""Cost of the deterministic mode (FGNN_DETERMINISTIC): default vs deterministic, as one JSON document.

  python tools/deterministic_bench.py --out deterministic.json

Measures, on cuda:0, with the card's name and power limit read in the same run, fp16, 4 blocks of depth 3, ErdosRenyi
p = 0.2 pairs drawn on the device:
  * cfg2 training step: training.train_step_flat on 128 pairs of n = 200, C = 32;
  * cfg3 forward: Siamese_Node_Exp.loss_and_accuracy (embedder + fused head, no grad) on 64 pairs of n = 500, C = 64;
  * one N = 2048 forward: the embeddings of one graph of n = 2048, C = 64.
The mode is switched with the FGNN_DETERMINISTIC environment variable (torch's own deterministic settings, which also
fill new tensors, stay off: the numbers are the library's cost).  The two arms are alternated for --rounds rounds; each
round times a window of repeated calls between CUDA events lasting at least --min-window seconds; medians are reported.
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from tools.head_train_bench import card, timed  # noqa: E402


def mode(det):
    def wrap(fn):
        def run():
            os.environ["FGNN_DETERMINISTIC"] = "1" if det else "0"
            return fn()
        return run
    return wrap


def alternate(fn, rounds, min_window):
    """fn under both modes, alternated round by round: {mode: (median ms, [ms per round])}."""
    arms = {"default": mode(False)(fn), "deterministic": mode(True)(fn)}
    times = {k: [] for k in arms}
    for f in arms.values():
        for _ in range(2):
            f()
    torch.cuda.synchronize()
    for _ in range(rounds):
        for k, f in arms.items():
            times[k].append(timed(f, min_window))
    out = {k: {"median_ms": statistics.median(v), "rounds_ms": v} for k, v in times.items()}
    out["overhead"] = out["deterministic"]["median_ms"] / out["default"]["median_ms"] - 1.0
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--min-window", type=float, default=1.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import graph_neural_net_b200 as pkg
    from graph_neural_net_b200 import _ops
    from graph_neural_net_b200.training import FlatAdam, train_step_flat

    dev = torch.device("cuda:0")

    def model(c):
        node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=4,
                        in_features=c, out_features=c, depth_of_mlp=3)
        torch.manual_seed(3787)
        return pkg.models.Siamese_Node_Exp(2, node_emb).to(dev).set_precision("fp16")

    def batch(pairs, n):
        a1, a2 = _ops.generate_pairs(0, pairs, n, 0.2, 0.1, 1234, None, dev)
        return {"input": _ops.features_from_adjacency(a1, None)}, {"input": _ops.features_from_adjacency(a2, None)}

    res = {"card": card(), "rounds": args.rounds, "min_window_s": args.min_window}
    m2 = model(32)
    opt = FlatAdam(m2.parameters(), lr=m2.lr)
    x1, x2 = batch(128, 200)
    res["cfg2_train_step_flat"] = alternate(lambda: train_step_flat(m2, opt, x1, x2), args.rounds, args.min_window)
    del m2, opt, x1, x2
    _ops.L.release_workspaces()
    torch.cuda.empty_cache()
    m3 = model(64)
    x1, x2 = batch(64, 500)

    @torch.no_grad()
    def fwd3():
        loss, ok, rows = m3.loss_and_accuracy(x1, x2)
        return loss

    res["cfg3_forward"] = alternate(fwd3, args.rounds, args.min_window)
    del x1, x2
    xb, _ = batch(1, 2048)

    @torch.no_grad()
    def fwd_big():
        return m3.embed(xb)

    res["n2048_forward"] = alternate(fwd_big, args.rounds, args.min_window)
    os.environ.pop("FGNN_DETERMINISTIC", None)
    doc = json.dumps(res, indent=1)
    print(doc)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(doc)


if __name__ == "__main__":
    main()
