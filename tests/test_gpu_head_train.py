"""GPU tests of the fused head's training form (fgnn_head_fwd_train / fgnn_head_bwd, _ops.HeadFunction,
training.train_step_flat(fused_head=True)): gradients against fp64 autograd and against the CUDA-core path
(ScoresFunction + CrossEntropyIdentityFunction), bitwise agreement with the inference head, determinism, memory
without any (G,N,N) tensor, the end-to-end training step, and the limits."""
import numpy as np
import pytest
import torch

import graph_neural_net_b200 as pkg
from graph_neural_net_b200 import _lib as L
from graph_neural_net_b200 import _ops
from graph_neural_net_b200.maskedtensors import maskedtensor as mt
from graph_neural_net_b200.toolbox.losses import triplet_loss
from graph_neural_net_b200.training import FlatAdam, train_step_flat
from oracle import fgnn_oracle as O
from tests.helpers import load_golden, rel_fro, state_dict_of

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# (G, C, N, sizes or None)
SHAPES = [(3, 32, 50, None), (2, 64, 500, None), (2, 128, 1000, None), (2, 20, 77, None),
          (2, 32, 4096, [4096, 2049]), (5, 16, 300, [300, 129, 40, 1, 257])]


def make_inputs(G, C, N, sizes, seed):
    """e1 = e2 + noise: the scores peak on the diagonal (s_ii ~ 4).  Entries beyond n_g hold garbage, which every
    head must ignore."""
    gen = torch.Generator().manual_seed(seed)
    e2 = torch.randn(G, C, N, generator=gen) * (4.0 / C) ** 0.5
    e1 = e2 + 0.5 * torch.randn(G, C, N, generator=gen) * (4.0 / C) ** 0.5
    coef = torch.rand(G, generator=gen) * 2.0 + 0.25               # per-graph d loss / d ce_sum, all different
    coef[0] = 1.0 / (G * N)                                          # 1 / #rows: coef p is below fp16's normal range
    n = sizes or [N] * G
    return e1, e2, coef, n


def fp64_reference(e1, e2, coef, n):
    """Gradients of sum_g coef_g ce_sum[g] by torch fp64 autograd on the valid blocks; lse of every valid row."""
    G, C, N = e1.shape
    a = e1.double().clone().requires_grad_(True)
    b = e2.double().clone().requires_grad_(True)
    total = 0.0
    lses = torch.zeros(G, N, dtype=torch.float64)
    for g in range(G):
        s = a[g, :, :n[g]].T @ b[g, :, :n[g]]
        lse = torch.logsumexp(s, dim=1)
        lses[g, :n[g]] = lse.detach()
        total = total + coef[g].double() * (lse - s.diagonal()).sum()
    total.backward()
    return a.grad, b.grad, lses


def fused(e1, e2, coef, n, prec):
    """HeadFunction forward + backward with upstream gradient coef."""
    x1 = e1.to(DEV).requires_grad_(True)
    x2 = e2.to(DEV).requires_grad_(True)
    n_dev = torch.tensor(n, dtype=torch.int32, device=DEV)
    ce, correct = _ops.HeadFunction.apply(x1, x2, n_dev, prec)
    ce.backward(coef.to(DEV))
    return ce.detach(), correct, x1.grad, x2.grad


def check_padding(g, n):
    for k, nk in enumerate(n):
        assert torch.count_nonzero(g[k, :, nk:]) == 0


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("G,C,N,sizes", SHAPES)
def test_head_gradients_match_fp64_and_cuda_core(G, C, N, sizes, prec):
    e1, e2, coef, n = make_inputs(G, C, N, sizes, seed=G * 1000 + C + N)
    r1, r2, _ = fp64_reference(e1, e2, coef, n)
    _, _, d1, d2 = fused(e1, e2, coef, n, prec)
    for g_ in (d1, d2):
        assert torch.isfinite(g_).all()
        check_padding(g_, n)
    err1, err2 = rel_fro(d1.cpu(), r1), rel_fro(d2.cpu(), r2)
    # the CUDA-core path on the same inputs
    y1 = e1.to(DEV).requires_grad_(True)
    y2 = e2.to(DEV).requires_grad_(True)
    n_dev = torch.tensor(n, dtype=torch.int32, device=DEV)
    ce_ref, _ = _ops.CrossEntropyIdentityFunction.apply(_ops.ScoresFunction.apply(y1, y2, n_dev), n_dev)
    ce_ref.backward(coef.to(DEV))
    c1, c2 = rel_fro(d1.cpu(), y1.grad.cpu()), rel_fro(d2.cpu(), y2.grad.cpu())
    print(f"head bwd {prec} G={G} C={C} N={N}: vs fp64 de1 {err1:.2e} de2 {err2:.2e}; vs CUDA-core de1 {c1:.2e} de2 {c2:.2e}")
    assert err1 <= 1e-4 and err2 <= 1e-4
    assert c1 <= 1e-4 and c2 <= 1e-4


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("G,C,N,sizes", [SHAPES[0], SHAPES[3], SHAPES[4], SHAPES[5]])
def test_training_forward_matches_inference_head(G, C, N, sizes, prec):
    e1, e2, coef, n = make_inputs(G, C, N, sizes, seed=7 + N)
    _, _, lse_ref = fp64_reference(e1, e2, coef, n)
    a, b = e1.to(DEV), e2.to(DEV)
    n_dev = torch.tensor(n, dtype=torch.int32, device=DEV)
    ce_inf, ok_inf, _ = _ops.head_fused(a, b, n_dev, prec)
    lib = L.get_lib()
    Cp = (C + 15) // 16 * 16
    ap = torch.nn.functional.pad(a, (0, 0, 0, Cp - C)).contiguous()
    bp = torch.nn.functional.pad(b, (0, 0, 0, Cp - C)).contiguous()
    ce = torch.empty(G, device=DEV)
    ok = torch.empty(G, device=DEV, dtype=torch.int32)
    lse = torch.full((G, N), float("nan"), device=DEV)
    ws = L.workspace(DEV, lib.fgnn_head_workspace_bytes(G, N))
    L.check(lib.fgnn_head_fwd_train(L.PRECISIONS[prec], L.ptr(ap), L.ptr(bp), L.ptr(ce), L.ptr(ok), L.ptr(lse), G, Cp, N,
                                    L.ptr(n_dev), L.ptr(ws), ws.numel(), L.stream_ptr(DEV)), "fgnn_head_fwd_train")
    assert torch.equal(ce, ce_inf) and torch.equal(ok, ok_inf)
    err = float((lse.double().cpu() - lse_ref).abs().max())
    print(f"row lse {prec} G={G} C={C} N={N}: max abs err vs fp64 {err:.2e}")
    assert err <= 1e-5 * max(1.0, float(lse_ref.abs().max()))
    for k, nk in enumerate(n):
        assert torch.count_nonzero(lse[k, nk:]) == 0


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
def test_head_backward_is_deterministic(prec):
    e1, e2, coef, n = make_inputs(5, 16, 300, [300, 129, 40, 1, 257], seed=99)
    _, _, a1, a2 = fused(e1, e2, coef, n, prec)
    _, _, b1, b2 = fused(e1, e2, coef, n, prec)
    assert torch.equal(a1, b1) and torch.equal(a2, b2)


def test_head_training_needs_no_quadratic_memory():
    G, C, N = 8, 64, 4096
    e1, e2, coef, n = make_inputs(G, C, N, None, seed=5)
    x1 = e1.to(DEV).requires_grad_(True)
    x2 = e2.to(DEV).requires_grad_(True)
    cf = coef.to(DEV)
    L.workspace(DEV, L.get_lib().fgnn_head_workspace_bytes(G, N))
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated(DEV)
    torch.cuda.reset_peak_memory_stats(DEV)
    ce, _ = _ops.HeadFunction.apply(x1, x2, None, "fp16")
    ce.backward(cf)
    torch.cuda.synchronize()
    extra = torch.cuda.max_memory_allocated(DEV) - base
    print(f"fused head fwd + bwd G={G} N={N} C={C}: peak above the inputs {extra / 2**20:.1f} MiB")
    assert extra < G * N * N * 4


def feats(W):
    return torch.stack([O.adjacency_to_features(torch.from_numpy(w.astype(np.float32))) for w in W])


def step_pair(make_model, x1, x2):
    """First-step (loss, correct, rows) and flat gradients of both arms, from identical copies of the model."""
    out = {}
    for fh in (False, True):
        _ops.GradScale.log2, _ops.GradScale._good = 9, 0
        model = make_model()
        opt = FlatAdam(model.parameters(), lr=model.lr)
        res = train_step_flat(model, opt, x1, x2, fused_head=fh)
        out[fh] = (res, opt.flat_g[:opt.n].clone())
    return out


def compare_first_step(out, label):
    (la, ga), (lb, gb) = out[False], out[True]
    gerr = rel_fro(gb.cpu(), ga.cpu())
    print(f"train_step_flat {label}: loss {la[0]:.7f} vs fused {lb[0]:.7f}; flat grad rel err {gerr:.2e}")
    assert abs(la[0] - lb[0]) <= 1e-5 * max(1.0, abs(la[0]))
    assert la[1:] == lb[1:]
    assert gerr <= 1e-3


def test_train_step_fused_head_golden():
    z = load_golden("cfg1_er50_c32")
    n, c, nb, depth, _ = [int(v) for v in z["meta"]]
    node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=nb,
                    in_features=c, out_features=c, depth_of_mlp=depth)

    def make_model():
        m = pkg.models.Siamese_Node_Exp(2, dict(node_emb))
        m.load_state_dict(state_dict_of(z))
        return m.to(DEV).set_precision("fp16")

    x1, x2 = {"input": feats(z["W1"]).to(DEV)}, {"input": feats(z["W2"]).to(DEV)}
    compare_first_step(step_pair(make_model, x1, x2), "cfg1 fp16")
    _ops.GradScale.log2, _ops.GradScale._good = 9, 0
    model = make_model()
    opt = FlatAdam(model.parameters(), lr=model.lr)
    losses = [train_step_flat(model, opt, x1, x2, fused_head=True)[0] for _ in range(6)]
    print("fused-head train_step_flat losses", [round(v, 4) for v in losses])
    assert losses[-1] < losses[0]


@pytest.mark.parametrize("cst", [False, True])
def test_train_step_fused_head_ragged(cst):
    gen = torch.Generator().manual_seed(41)
    sizes = [50, 23, 37, 64, 130]
    sd = O.xavier_state_dict(2, 32, 3, 3, gen, randomize_gn=True)
    node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=3,
                    in_features=32, out_features=32, depth_of_mlp=3, constant_n_vertices=cst)
    pairs = [O.synthetic_pair(s, 0.3, 0.1, gen) for s in sizes]

    def make_model():
        m = pkg.models.Siamese_Node_Exp(2, dict(node_emb))
        m.load_state_dict(sd)
        return m.to(DEV).set_precision("fp16")

    x1 = {"input": mt.from_list([p[0] for p in pairs], dims=(1, 2)).to(DEV)}
    x2 = {"input": mt.from_list([p[1] for p in pairs], dims=(1, 2)).to(DEV)}
    compare_first_step(step_pair(make_model, x1, x2), f"ragged constant_n={cst}")


def test_train_step_leaves_no_gradient_sink_behind():
    """The flat step publishes its model's parameter addresses as the sink of the 16-bit backward; left behind after
    the step, they captured the gradients of a later model whose parameters reuse those addresses (its p.grad stayed
    None).  Either head: the sink is empty after the step and a fresh model trained by plain autograd gets every
    gradient."""
    z = load_golden("cfg1_er50_c32")
    n, c, nb, depth, _ = [int(v) for v in z["meta"]]
    node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=nb,
                    in_features=c, out_features=c, depth_of_mlp=depth)

    def make_model():
        m = pkg.models.Siamese_Node_Exp(2, dict(node_emb))
        m.load_state_dict(state_dict_of(z))
        return m.to(DEV).set_precision("fp16")

    x1, x2 = {"input": feats(z["W1"]).to(DEV)}, {"input": feats(z["W2"]).to(DEV)}
    for fh in (False, True):
        model = make_model()
        opt = FlatAdam(model.parameters(), lr=model.lr)
        train_step_flat(model, opt, x1, x2, fused_head=fh)
        assert not _ops.GRAD_SINK
        del model, opt
        fresh = make_model()
        triplet_loss("mean")(fresh(x1, x2)).backward()
        missing = [k for k, p in fresh.named_parameters() if p.grad is None]
        assert not missing, missing


def test_head_training_limits_fail_loudly():
    e = torch.zeros(2, 32, 64, device=DEV)
    with pytest.raises(L.FgnnError, match="fp32"):
        _ops.HeadFunction.apply(e, e, None, "fp32")
    big = torch.zeros(1, 16, 4097, device=DEV)
    with pytest.raises(L.FgnnError, match="4096"):
        _ops.HeadFunction.apply(big, big, None, "fp16")
    wide = torch.zeros(1, 144, 64, device=DEV)
    with pytest.raises(L.FgnnError, match="at most 128"):
        _ops.HeadFunction.apply(wide, wide, None, "fp16")
    lib = L.get_lib()
    out = torch.zeros(1, 144, 64, device=DEV)
    st = lib.fgnn_head_bwd(L.FP16, L.ptr(wide), L.ptr(wide), L.ptr(out), L.ptr(out), L.ptr(out), L.ptr(out), 1, 144, 64,
                           None, None, 0, L.stream_ptr(DEV))
    assert st != 0 and "at most 128" in lib.fgnn_last_error().decode()
    st = lib.fgnn_head_bwd(L.FP32, L.ptr(e), L.ptr(e), L.ptr(out), L.ptr(out), L.ptr(out), L.ptr(out), 2, 32, 64,
                           None, None, 0, L.stream_ptr(DEV))
    assert st != 0
    node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=2,
                    in_features=16, out_features=16, depth_of_mlp=2)
    model = pkg.models.Siamese_Node_Exp(2, node_emb).to(DEV).set_precision("fp32")
    opt = FlatAdam(model.parameters(), lr=1e-3)
    x = {"input": torch.zeros(1, 2, 8, 8, device=DEV)}
    with pytest.raises(L.FgnnError, match="fp32"):
        train_step_flat(model, opt, x, x, fused_head=True)
