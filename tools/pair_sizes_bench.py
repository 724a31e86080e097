"""Time the fused tensor-core head (forward + backward, _ops.HeadFunction, fp16) and the device linear assignment on
square pairs against rectangular pairs of the same n1 * n2, as one JSON document on stdout.  CUDA events around
`--iters` calls after a warm-up; inputs are random, so the LAP times are those of untrained-model scores."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from graph_neural_net_b200 import _ops  # noqa: E402
from graph_neural_net_b200.toolbox.metrics import linear_assignment  # noqa: E402


def timed(fn, iters):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def head_case(G, C, N1, N2, iters):
    gen = torch.Generator(device="cuda").manual_seed(N1 * 7 + N2)
    e1 = torch.randn(G, C, N1, device="cuda", generator=gen).requires_grad_(True)
    e2 = torch.randn(G, C, N2, device="cuda", generator=gen).requires_grad_(True)

    def step():
        _ops.HeadFunction.apply(e1, e2, None, "fp16")[0].sum().backward()
    return timed(step, iters)


def lap_case(G, N1, N2, iters):
    gen = torch.Generator(device="cuda").manual_seed(N1 * 3 + N2)
    s = torch.randn(G, N1, N2, device="cuda", generator=gen) * 3
    return timed(lambda: linear_assignment(s), iters)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    out = {"gpu": gpu, "head_fwd_bwd_fp16_ms": [], "lap_ms": []}
    # two passes over the shapes; the second is reported, so that no shape pays for the clocks ramping up
    for rep in range(2):
        head = [{"G": 16, "C": 64, "N1": N1, "N2": N2, "ms": round(head_case(16, 64, N1, N2, args.iters), 4)}
                for (N1, N2) in [(1024, 1024), (512, 2048), (2048, 512), (4096, 4096), (2048, 4096)]]
        lap = [{"G": 16, "N1": N1, "N2": N2, "ms": round(lap_case(16, N1, N2, max(2, args.iters // 4)), 3)}
               for (N1, N2) in [(512, 512), (256, 1024), (1024, 256)]]
    out["head_fwd_bwd_fp16_ms"], out["lap_ms"] = head, lap
    print(json.dumps(out))


if __name__ == "__main__":
    main()
