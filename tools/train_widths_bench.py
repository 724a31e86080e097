"""Time one training step of an embedder whose widths the 16-bit path zero-pads, against its uniform twin and fp32.

  python tools/train_widths_bench.py --out train_widths.json

On cuda:0, with the card's name and power limit read in the same run: training.train_step_flat at cfg2 (128 ErdosRenyi
p = 0.2 pairs of n = 200 drawn on the device, 4 blocks of depth 3) for
  * in_features = 32, out_features = 16 in fp16 (run zero-padded to C = 32),
  * its uniform twin, in = out = 32, in fp16,
  * the first model in fp32 (CUDA-core operators).
The arms are alternated for --rounds rounds of windows of at least --min-window seconds (head_train_bench.py); the
medians are reported as ms per step and pairs per second.
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from head_train_bench import ROOT, alternate, card  # noqa: E402,F401  (ROOT: the repository is on sys.path)

import torch  # noqa: E402


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True, help="JSON file to write")
    ap.add_argument("--min-window", type=float, default=2.0)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("train_widths_bench.py measures the GPU: no CUDA device")

    import graph_neural_net_b200 as pkg
    from graph_neural_net_b200 import _ops
    from graph_neural_net_b200.training import train_step_flat, FlatAdam

    dev = torch.device("cuda:0")
    pairs, n = 128, 200
    res = {"card": card(), "torch": torch.__version__, "time": time.strftime("%Y-%m-%dT%H:%M:%S"), "pairs": pairs, "n": n,
           "blocks": 4, "depth": 3}
    a1, a2 = _ops.generate_pairs(0, pairs, n, 0.2, 0.1, 1234, None, dev)
    b1, b2 = {"input": _ops.features_from_adjacency(a1, None)}, {"input": _ops.features_from_adjacency(a2, None)}
    arms = {}
    for label, in_f, out_f, prec in (("in32_out16_fp16", 32, 16, "fp16"), ("uniform32_fp16", 32, 32, "fp16"),
                                     ("in32_out16_fp32", 32, 16, "fp32")):
        torch.manual_seed(0)
        node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=4,
                        in_features=in_f, out_features=out_f, depth_of_mlp=3)
        model = pkg.models.Siamese_Node_Exp(2, node_emb).to(dev).set_precision(prec)
        opt = FlatAdam(model.parameters(), lr=model.lr)
        arms[label] = (lambda m=model, o=opt: train_step_flat(m, o, b1, b2))
    t = alternate(arms, args.rounds, args.min_window)
    res["steps"] = {k: {"ms": v[0], "pairs_per_s": pairs / (v[0] * 1e-3), "ms_rounds": v[1]} for k, v in t.items()}
    res["card_after"] = card()
    print(json.dumps(res["steps"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
