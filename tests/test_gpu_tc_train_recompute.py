"""GPU tests of 16-bit training in passes (fgnn_embed_fwd_train / fgnn_embed_bwd cut into passes whose activations the
backward re-derives from the input planes).

A batch is cut into passes when its one-pass workspace exceeds FGNN_TC_TRAIN_WS_GB (default: half the device's
memory), so the tests force passes with FGNN_TC_TRAIN_WS_GB=0 and set them with FGNN_TC_CHUNK; the one-pass runs
("keep-all") they are compared with set a threshold no batch here reaches.  Every pass runs the same kernels per graph,
and the forward is deterministic: a batch that fits one pass gives the same embeddings bit for bit whatever the
threshold (measured), and its backward re-runs nothing.  What differs with several passes is how many graphs share a
launch.  That changes how the conv-chain kernel's CTAs split the (graph, tile) work, so the GraphNorm statistics are
summed in another order and 16-bit activations round differently from the first block on.  The inference path shows
the same when FGNN_TC_CHUNK cuts a ragged batch into passes (2.0e-3 to 3.0e-3 on the embeddings of the batches below).
Weight-gradient reductions are fp32 atomics in any order (a few 1e-7 between two runs on the same passes).
"""
import numpy as np
import pytest
import torch

import graph_neural_net_b200 as pkg
from graph_neural_net_b200 import _ops
from graph_neural_net_b200.maskedtensors import maskedtensor as mt
from graph_neural_net_b200.toolbox.losses import triplet_loss
from oracle import fgnn_oracle as O
from tests.helpers import load_golden, state_dict_of, rel_fro
from tests.test_gpu_tc_train import EMUL_TOL, REF_TOL, TDT, build_model, compare_grads, feats, unpack_adj

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def use_plan(monkeypatch, recompute, chunk=None):
    monkeypatch.setenv("FGNN_TC_TRAIN_WS_GB", "0" if recompute else "100000")
    if chunk is None:
        monkeypatch.delenv("FGNN_TC_CHUNK", raising=False)
    else:
        monkeypatch.setenv("FGNN_TC_CHUNK", str(chunk))


def train_once(model, x1, x2):
    """One siamese forward + backward with the reference's mean loss: (loss, [e1, e2], {name: grad})."""
    _ops.GRAD_SINK.clear()      # a flat trainer of an earlier test may have left its sink behind: gradients go to p.grad
    for p in model.parameters():
        p.grad = None
    embs = []
    embed = model.embed
    model.embed = lambda x: embs.append(embed(x)) or embs[-1]      # keep the embeddings the scores are made of
    try:
        loss = triplet_loss("mean")(model(x1, x2))
    finally:
        del model.embed
    loss.backward()
    embs = [(e.tensor.rename(None) if isinstance(e, mt.MaskedTensor) else e).detach().cpu() for e in embs]
    return float(loss.detach()), embs, {k: p.grad.detach().cpu().clone() for k, p in model.named_parameters()}


def compare_plans(label, rc, ka, tols):
    """Two plans on the same batch: loss (relative), embeddings, all parameter gradients together."""
    loss_tol, emb_tol, grad_tol = tols
    dl = abs(rc[0] - ka[0]) / max(1.0, abs(ka[0]))
    de = max(rel_fro(a, b) for a, b in zip(rc[1], ka[1]))
    a = torch.cat([rc[2][k].flatten() for k in ka[2]])
    b = torch.cat([ka[2][k].flatten() for k in ka[2]])
    dg = rel_fro(a, b)
    worst = max(ka[2], key=lambda k: rel_fro(rc[2][k], ka[2][k]))
    print(f"PARITY {label}: loss {dl:.3e}, embeddings {de:.3e}, all parameters {dg:.3e} "
          f"(worst tensor {worst} {rel_fro(rc[2][worst], ka[2][worst]):.3e})")
    assert dl < loss_tol, dl
    assert de < emb_tol, de
    assert dg < grad_tol, dg


# recompute vs keep-all, (loss relative, embeddings, all parameter gradients together).  Goldens: measured 0, 0 and
# <= 2.7e-7 over the four cases (at most 100 tiles a launch: one per CTA on either plan); the bound leaves room for
# the fp32 atomics of the weight gradients.
GOLDEN_PLAN_TOL = (1e-6, 1e-6, 1e-6)
# Ragged batch [130, 64, 50, 37, 23], passes of 2: measured 2.0e-6, 3.1e-3, 2.9e-2 (constant_n False) and 6.7e-7,
# 3.6e-3, 3.0e-2 (True), the same on repeated runs.  Keep-all runs the 5 graphs in one launch (772 conv-chain tiles),
# a pass 2 graphs at most (388 tiles); cutting this batch into passes moves the inference path's embeddings by
# 2.2e-3 to 3.0e-3, and both plans are as far from the fp32 path (gradients: recompute 1.0e-1 / 1.4e-1, keep-all
# 1.1e-1 / 1.4e-1).
RAGGED_PLAN_TOL = (2.5e-6, 4.3e-3, 3.6e-2)
# recompute in passes of 1 vs passes of 2 on that batch: measured 0, 0, <= 3.8e-7
RAGGED_PASSES_TOL = (1e-6, 1e-6, 1e-6)


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("name", ["cfg1_er50_c32", "cfg2_er200_c32"])
def test_recompute_gradients_match_oracles_and_keep_all(name, prec, monkeypatch):
    """cfg1 (4 pairs) runs as 4 passes of one graph, each re-derived in backward; cfg2 (1 pair) as one pass, which the
    backward does not re-run (the same work as the one-pass run it is compared with)."""
    z = load_golden(name)
    n = int(z["meta"][0])
    if "W1" in z:
        x1, x2 = feats(z["W1"]).to(DEV), feats(z["W2"]).to(DEV)
    else:
        x1, x2 = feats(unpack_adj(z["W1_bits"], n)).to(DEV), feats(unpack_adj(z["W2_bits"], n)).to(DEV)
    use_plan(monkeypatch, False)
    ka = train_once(build_model(z, prec), {"input": x1}, {"input": x2})
    use_plan(monkeypatch, True, chunk=1)
    model = build_model(z, prec)
    rc = train_once(model, {"input": x1}, {"input": x2})
    compare_plans(f"recompute vs keep-all {name} {prec}", rc, ka, GOLDEN_PLAN_TOL)
    depth, nb = int(z["meta"][3]), int(z["meta"][2])
    eloss, egrads = O.emulated16_loss_and_grads(x1.cpu(), x2.cpu(), state_dict_of(z), TDT[prec])
    assert abs(rc[0] - eloss) < 2e-4 * max(1.0, abs(eloss)), (rc[0], eloss)
    ref = {k[5:]: z[k] for k in z if k.startswith("grad/")}
    try:
        compare_grads(model, egrads, EMUL_TOL[prec], f"{name} {prec} recompute vs emulated-16-bit-forward autograd", depth, nb)
    finally:
        compare_grads(model, ref, REF_TOL[prec], f"{name} {prec} recompute vs reference fp32 autograd", depth, nb)


def test_backward_re_runs_the_forward_only_for_several_passes(monkeypatch):
    """Kernel launches of each fgnn_embed_bwd call (x1's and x2's) on cfg1's 4 pairs: with FGNN_TC_TRAIN_WS_GB=0 and
    FGNN_TC_CHUNK >= G the batch is one pass whose activations the forward left in place, so the backward launches
    exactly what it does below the threshold; in two passes it launches more (each pass's forward again)."""
    z = load_golden("cfg1_er50_c32")
    x1, x2 = feats(z["W1"]).to(DEV), feats(z["W2"]).to(DEV)
    G = x1.shape[0]
    lib = pkg.get_lib()
    embed_bwd, counts = lib.fgnn_embed_bwd, []

    def counted(*args):      # runs on autograd's thread: the launch counter is thread-local
        lib.fgnn_reset_launch_count()
        status = embed_bwd(*args)
        counts.append(lib.fgnn_launch_count())
        return status

    monkeypatch.setattr(lib, "fgnn_embed_bwd", counted)

    def launches(recompute, chunk):
        counts.clear()
        use_plan(monkeypatch, recompute, chunk)
        train_once(build_model(z, "fp16"), {"input": x1}, {"input": x2})
        assert len(counts) == 2, counts
        return list(counts)

    one_pass = launches(False, None)
    assert launches(True, G) == one_pass
    assert launches(True, 2 * G) == one_pass
    two = launches(True, G // 2)
    print(f"PARITY fgnn_embed_bwd launches: one pass {one_pass}, two passes {two}")
    assert all(t > o for t, o in zip(two, one_pass)), (two, one_pass)


def ragged_runs(sizes, cst, plans, monkeypatch):
    """{label: train_once result} for a 3-block, width-32 model on a ragged batch of `sizes`; plans: (label, precision,
    recompute, chunk)."""
    gen = torch.Generator().manual_seed(31)
    sd = O.xavier_state_dict(2, 32, 3, 3, gen, randomize_gn=True)
    node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=3,
                    in_features=32, out_features=32, depth_of_mlp=3, constant_n_vertices=cst)
    pairs = [O.synthetic_pair(s, 0.3, 0.1, gen) for s in sizes]
    x1 = mt.from_list([p[0] for p in pairs], dims=(1, 2)).to(DEV)
    x2 = mt.from_list([p[1] for p in pairs], dims=(1, 2)).to(DEV)
    runs = {}
    for label, prec, recompute, chunk in plans:
        use_plan(monkeypatch, recompute, chunk)
        model = pkg.models.Siamese_Node_Exp(2, dict(node_emb))
        model.load_state_dict(sd)
        model = model.to(DEV).set_precision(prec)
        runs[label] = train_once(model, {"input": x1}, {"input": x2}) + (model,)
    return runs


@pytest.mark.parametrize("cst", [False, True])
def test_recompute_ragged_passes_match_keep_all(cst, monkeypatch):
    """Passes of two graphs, [130, 64] then [50, 37], [23]: the smaller graphs of a later pass run in planes an earlier
    pass filled further (every pass zeroes them again).  Passes of one graph cut the batch differently and must
    agree bit for bit in the forward."""
    runs = ragged_runs([130, 64, 50, 37, 23], cst, (("keep-all", "fp16", False, None), ("passes of 1", "fp16", True, 1),
                                                    ("recompute", "fp16", True, 2)), monkeypatch)
    compare_plans(f"recompute vs keep-all ragged constant_n={cst} fp16", runs["recompute"], runs["keep-all"],
                  RAGGED_PLAN_TOL)
    compare_plans(f"recompute in passes of 2 vs passes of 1 ragged constant_n={cst} fp16", runs["recompute"],
                  runs["passes of 1"], RAGGED_PASSES_TOL)


@pytest.mark.parametrize("cst", [False, True])
def test_recompute_ragged_gradients_match_fp32_path(cst, monkeypatch):
    """The batch and envelope of test_tc_training_ragged_gradients_match_fp32_path, on the recompute plan in passes
    [50, 23], [37, 64], [130]: fp16 tcgen05 gradients vs the fp32 CUDA operators' autograd."""
    runs = ragged_runs([50, 23, 37, 64, 130], cst, (("fp32", "fp32", False, None), ("recompute", "fp16", True, 2)),
                       monkeypatch)
    assert abs(runs["recompute"][0] - runs["fp32"][0]) < 5e-3 * max(1.0, abs(runs["fp32"][0]))
    compare_grads(runs["recompute"][3], {k: g.numpy() for k, g in runs["fp32"][2].items()}, (3e-1, 1e-1, 0.995, None),
                  f"ragged constant_n={cst} fp16 recompute vs fp32 CUDA", 3)


def cfg3_model(seed=64):
    gen = torch.Generator().manual_seed(seed)
    sd = O.xavier_state_dict(2, 64, 4, 3, gen)
    node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=4,
                    in_features=64, out_features=64, depth_of_mlp=3)
    m = pkg.models.Siamese_Node_Exp(2, node_emb)
    m.load_state_dict(sd)
    return m.to(DEV).set_precision("fp16")


def cfg3_inputs(pairs=64, n=500, seed=500):
    a1, a2 = _ops.generate_pairs(0, pairs, n, 0.2, 0.1, seed, None, torch.device(DEV))      # ErdosRenyi, p = 0.2
    return _ops.features_from_adjacency(a1, None), _ops.features_from_adjacency(a2, None)


def test_cfg3_training_step_fits_with_default_threshold(monkeypatch):
    """64 pairs of n = 500, C = 64, 4 blocks of depth 3: 107 GB per embedder call on keep-all, twice per step, which no
    single device holds.  With the default threshold the step runs on the recompute plan."""
    from graph_neural_net_b200.training import train_step_flat, FlatAdam
    for v in ("FGNN_TC_TRAIN_WS_GB", "FGNN_TC_WS_GB", "FGNN_TC_CHUNK"):
        monkeypatch.delenv(v, raising=False)
    model = cfg3_model()
    opt = FlatAdam(model.parameters(), lr=model.lr)
    x1, x2 = cfg3_inputs()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()          # model, optimiser, inputs, and whatever earlier tests keep cached
    torch.cuda.reset_peak_memory_stats()
    try:
        loss, ok, rows = train_step_flat(model, opt, {"input": x1}, {"input": x2})
        torch.cuda.synchronize()
    finally:
        _ops.GRAD_SINK.clear()
    step = torch.cuda.max_memory_allocated() - base
    total = torch.cuda.get_device_properties(0).total_memory
    print(f"PARITY cfg3 recompute training step: loss {loss:.6f}, correct {ok}/{rows}, peak allocated by the step "
          f"{step / 1e9:.2f} GB of {total / 1e9:.1f} GB")
    assert np.isfinite(loss) and rows == 64 * 500
    assert step < 41e9, step          # measured 34.2 GB: two 16.8 GB workspaces (107 GB each on keep-all)


def test_full_batch_gradient_is_the_sum_of_quarter_batches(monkeypatch):
    """The un-normalised gradient of 64 pairs on the recompute plan (the default threshold picks it) equals the sum of
    the gradients of its four 16-pair quarters, each on keep-all (27 GB per call).  Every call picks its own loss
    scale, so the two differ by 16-bit rounding only."""
    for v in ("FGNN_TC_TRAIN_WS_GB", "FGNN_TC_WS_GB", "FGNN_TC_CHUNK"):
        monkeypatch.delenv(v, raising=False)
    _ops.GRAD_SINK.clear()
    model = cfg3_model()
    x1, x2 = cfg3_inputs()

    def grads(lo, hi):
        scores = model({"input": x1[lo:hi]}, {"input": x2[lo:hi]})
        ce, _ = _ops.CrossEntropyIdentityFunction.apply(scores, None)
        ce.sum().backward()
        return float(ce.sum().detach())

    model.zero_grad(set_to_none=True)
    full_loss = grads(0, 64)
    full = torch.cat([p.grad.detach().flatten() for p in model.parameters()])
    model.zero_grad(set_to_none=True)
    quarter_loss = sum(grads(q * 16, q * 16 + 16) for q in range(4))      # p.grad accumulates over the four calls
    summed = torch.cat([p.grad.detach().flatten() for p in model.parameters()])
    err = rel_fro(full.cpu(), summed.cpu())
    print(f"PARITY cfg3 full batch (recompute) vs sum of 4 quarter batches (keep-all): loss {abs(full_loss - quarter_loss) / quarter_loss:.3e}, "
          f"all parameters {err:.3e}")
    assert torch.isfinite(full).all()
    assert abs(full_loss - quarter_loss) < 3.2e-6 * quarter_loss      # measured 2.6e-6
    assert err < 3.6e-3, err                                          # measured 3.0e-3
