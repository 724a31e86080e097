"""16-bit training (and inference) of embedders whose widths are not a uniform 32 or 64.

The C library runs such a model zero-padded to C = 32 or 64: padded channels have zero weights, biases and GraphNorm
affine, so they are exactly zero everywhere.  The oracle is therefore the uniform TWIN of width C whose parameters are
the real ones zero-padded: its embeddings (inference and training forward) sliced to the real channels and its loss
must equal the model's bit for bit, and its gradients on the padded entries must be exact zeros.  Its gradients on the
real entries agree with the model's as closely as two backward passes of the twin agree with each other: the
weight-gradient reductions are fp32 atomics in any order, a few 1e-7 apart between two runs of the same model."""
import pytest
import torch

import graph_neural_net_b200 as pkg
from graph_neural_net_b200 import _lib as L
from graph_neural_net_b200 import _ops
from graph_neural_net_b200.maskedtensors import maskedtensor as mt
from graph_neural_net_b200.toolbox.losses import triplet_loss
from oracle import fgnn_oracle as O
from tests.test_gpu_tc_train import compare_grads

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CASES = [(48, 40, 2), (24, 32, 3), (32, 64, 3), (64, 20, 2), (16, 16, 3)]
SIZES = [50, 23, 37, 64, 130]
NB = 3


def node_emb(in_f, out_f, depth, cst=False):
    return dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=NB,
                in_features=in_f, out_features=out_f, depth_of_mlp=depth, constant_n_vertices=cst)


def make_model(in_f, out_f, depth, cst=False, seed=31):
    """The reference's init law with perturbed biases and GraphNorm affine (as the uniform-width parity tests use)."""
    model = pkg.models.Siamese_Node_Exp(2, node_emb(in_f, out_f, depth, cst))
    gen = torch.Generator().manual_seed(seed)
    model.load_state_dict(O.xavier_state_dict(2, in_f, NB, depth, gen, c_out=out_f, randomize_gn=True))
    return model


def pad_like(key, real, shape, C):
    """The real tensor zero-padded to the twin's shape: rows and columns at their own index, except the first conv of
    mlp3, which reads cat[mult, block input] -- its real columns [co, co + cin) sit at [C, C + cin) in the twin."""
    out = real.new_zeros(shape)
    if ".convs.0.weight" in key and "_mlp3." in key:
        co = real.shape[0]
        out[:co, :co] = real[:, :co]
        out[:co, C:C + real.shape[1] - co] = real[:, co:]
    elif real.dim() == 4:
        out[:real.shape[0], :real.shape[1]] = real
    else:
        out[:real.shape[0]] = real
    return out


def unpad(key, twin, real_shape, C):
    if ".convs.0.weight" in key and "_mlp3." in key:
        co = real_shape[0]
        return torch.cat([twin[:co, :co], twin[:co, C:C + real_shape[1] - co]], dim=1)
    if len(real_shape) == 4:
        return twin[:real_shape[0], :real_shape[1]]
    return twin[:real_shape[0]]


@pytest.fixture
def twin():
    """twin(model, in_f, out_f, depth, cst) -> (uniform model of width C with the zero-padded parameters, C)."""
    def build(model, in_f, out_f, depth, cst=False):
        C = 32 if max(in_f, out_f) <= 32 else 64
        tw = pkg.models.Siamese_Node_Exp(2, node_emb(C, C, depth, cst))
        real = dict(model.named_parameters())
        with torch.no_grad():
            for k, p in tw.named_parameters():
                p.copy_(pad_like(k, real[k].detach().to(p.device), p.shape, C))
        return tw.to(real[k].device).set_precision(model.precision), C
    return build


def ragged_pair(seed=7):
    gen = torch.Generator().manual_seed(seed)
    pairs = [O.synthetic_pair(s, 0.3, 0.1, gen) for s in SIZES]
    x1 = mt.from_list([p[0] for p in pairs], dims=(1, 2)).to(DEV)
    x2 = mt.from_list([p[1] for p in pairs], dims=(1, 2)).to(DEV)
    return x1, x2


def plain(e):
    return e.tensor.rename(None)


def head_loss(e1, e2, n_dev):
    """triplet_loss('mean') of e1^T e2 on (B, c, N) embeddings (the model's own 16-bit training head)."""
    s = _ops.ScoresFunction.apply(e1, e2, n_dev)
    ce, _ = _ops.CrossEntropyIdentityFunction.apply(s, n_dev)
    return ce.sum() / n_dev.to(torch.float32).sum()


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("in_f,out_f,depth", CASES)
def test_padded_widths_match_the_uniform_twin(in_f, out_f, depth, prec, twin):
    _ops.GRAD_SINK.clear()
    model = make_model(in_f, out_f, depth).to(DEV).set_precision(prec)
    tw, C = twin(model, in_f, out_f, depth)
    x1, x2 = ragged_pair()
    n_dev = x1.sizes_i32(DEV)
    net, tnet = model.node_embedder, tw.node_embedder
    with torch.no_grad():
        for x in (x1, x2):
            e, et = plain(net.forward_fused(x)), plain(tnet.forward_fused(x))
            assert e.shape == (len(SIZES), out_f, max(SIZES)) and et.shape[1] == C
            assert torch.equal(e, et[:, :out_f])
            assert not et[:, out_f:].any()
    e1, e2 = plain(net.forward_fused_train(x1)), plain(net.forward_fused_train(x2))
    t1, t2 = plain(tnet.forward_fused_train(x1)), plain(tnet.forward_fused_train(x2))
    assert torch.equal(e1.detach(), t1.detach()[:, :out_f]) and torch.equal(e2.detach(), t2.detach()[:, :out_f])
    loss = head_loss(e1, e2, n_dev)
    tloss = head_loss(t1[:, :out_f].contiguous(), t2[:, :out_f].contiguous(), n_dev)
    assert torch.equal(loss.detach(), tloss.detach())
    loss.backward()
    tloss.backward()
    treal = dict(tw.named_parameters())
    tgrads = {k: p.grad.clone() for k, p in treal.items()}
    for p in tw.parameters():                                          # the twin's run-to-run spread
        p.grad = None
    t1, t2 = plain(tnet.forward_fused_train(x1)), plain(tnet.forward_fused_train(x2))
    head_loss(t1[:, :out_f].contiguous(), t2[:, :out_f].contiguous(), n_dev).backward()
    mine, twin_a, twin_b = [], [], []
    for k, p in model.named_parameters():
        tg = tgrads[k]
        assert p.grad is not None and tg is not None, k
        mask = pad_like(k, torch.ones_like(p), tg.shape, C)
        assert not (tg * (1 - mask)).any(), k                      # padded entries: exact zeros
        mine.append(p.grad.flatten())
        twin_a.append(unpad(k, tg, p.shape, C).flatten())
        twin_b.append(unpad(k, treal[k].grad, p.shape, C).flatten())
    mine, twin_a, twin_b = torch.cat(mine), torch.cat(twin_a), torch.cat(twin_b)
    d_model = float((mine - twin_a).norm() / twin_a.norm())
    d_twin = float((twin_b - twin_a).norm() / twin_a.norm())
    print(f"PARITY {prec} in={in_f} out={out_f} depth={depth}: embeddings and loss {float(loss):.6f} bitwise equal to the "
          f"C={C} twin; gradients {d_model:.2e} from the twin's (two runs of the twin: {d_twin:.2e})")
    assert d_model <= 4 * d_twin + 2e-6, (d_model, d_twin)


@pytest.mark.parametrize("cst", [False, True])
@pytest.mark.parametrize("in_f,out_f,depth", CASES)
def test_padded_widths_train_like_the_fp32_path(in_f, out_f, depth, cst):
    """fp16 tcgen05 gradients vs the fp32 CUDA operators' autograd on a ragged batch.  The uniform models' envelope
    (test_tc_training_ragged_gradients_match_fp32_path: 3e-1 per tensor, 1e-1 together, cosine 0.995) holds for 8 of
    these 10 cases; measured worst on one B200: 3.96e-1 per tensor at (24, 32, 3) and 1.19e-1 together, cosine 0.9929 at
    (32, 64, 3), both constant_n=True.  Those models' gradients equal their zero-padded uniform twins' (the test
    above), so the spread is the 16-bit backward's on these random models, not the padding's."""
    _ops.GRAD_SINK.clear()
    sd = make_model(in_f, out_f, depth, cst).state_dict()
    x1, x2 = ragged_pair()
    grads, losses = {}, {}
    for prec in ("fp32", "fp16"):
        model = pkg.models.Siamese_Node_Exp(2, node_emb(in_f, out_f, depth, cst))
        model.load_state_dict(sd)
        model = model.to(DEV).set_precision(prec)
        loss = triplet_loss("mean")(model({"input": x1}, {"input": x2}))
        loss.backward()
        losses[prec] = float(loss.detach())
        grads[prec] = {k: p.grad.detach().cpu().numpy().copy() for k, p in model.named_parameters()}
        last = model
    print(f"PARITY loss in={in_f} out={out_f} depth={depth} constant_n={cst}: fp16 {losses['fp16']:.6f} "
          f"fp32 {losses['fp32']:.6f}")
    assert abs(losses["fp16"] - losses["fp32"]) < 5e-3 * max(1.0, abs(losses["fp32"]))
    compare_grads(last, grads["fp32"], (5e-1, 1.5e-1, 0.99, None),
                  f"in={in_f} out={out_f} depth={depth} constant_n={cst} fp16 vs fp32 CUDA", depth)


@pytest.mark.parametrize("fused_head", [False, True])
def test_flat_train_step_at_padded_widths(fused_head):
    from graph_neural_net_b200.training import train_step_flat, FlatAdam
    _ops.GRAD_SINK.clear()
    depth = 3
    model = make_model(24, 40, depth).to(DEV).set_precision("fp16")
    opt = FlatAdam(model.parameters(), lr=model.lr)
    x1, x2 = ragged_pair()
    names = [k for k, p in model.named_parameters() if p.requires_grad]
    losses = []
    for it in range(6):
        losses.append(train_step_flat(model, opt, {"input": x1}, {"input": x2}, fused_head=fused_head)[0])
        assert not _ops.GRAD_SINK
        assert float(opt.extras[3]) == 0.0, it                    # no gradient overflowed (nothing was zeroed)
        if it == 0:
            for k, g in zip(names, opt.grad_views):
                assert torch.isfinite(g).all(), k
                if not k.endswith(f"convs.{depth - 1}.bias"):      # cancels in GraphNorm: rounding noise around 0
                    assert float(g.abs().max()) > 0, k
    print(f"fp16 train_step_flat (fused_head={fused_head}) in=24 out=40 losses", [round(v, 4) for v in losses])
    assert losses[-1] < losses[0]


def test_recompute_plan_reproduces_keep_all_at_padded_widths(monkeypatch):
    _ops.GRAD_SINK.clear()
    model = make_model(24, 40, 3).to(DEV).set_precision("fp16")
    x1, x2 = ragged_pair()
    n_dev = x1.sizes_i32(DEV)
    net = model.node_embedder

    def run():
        model.zero_grad(set_to_none=True)
        e1, e2 = plain(net.forward_fused_train(x1)), plain(net.forward_fused_train(x2))
        loss = head_loss(e1, e2, n_dev)
        loss.backward()
        return [loss.detach(), e1.detach().clone(), e2.detach().clone()], torch.cat([p.grad.flatten() for p in model.parameters()])

    monkeypatch.delenv("FGNN_TC_CHUNK", raising=False)
    monkeypatch.setenv("FGNN_TC_TRAIN_WS_GB", "1000")
    ref, gref = run()
    _, gref2 = run()                                                    # run-to-run spread of the atomics
    monkeypatch.setenv("FGNN_TC_TRAIN_WS_GB", "0")
    monkeypatch.setenv("FGNN_TC_CHUNK", str(len(SIZES)))             # one recompute pass
    got, g = run()
    assert all(torch.equal(a, b) for a, b in zip(ref, got))             # loss and embeddings bit for bit
    d, d_ka = float((g - gref).norm() / gref.norm()), float((gref2 - gref).norm() / gref.norm())
    print(f"PARITY recompute (one pass) vs keep-all in=24 out=40: gradients {d:.2e} (two keep-all runs: {d_ka:.2e})")
    assert d <= 4 * d_ka + 2e-6, (d, d_ka)


@pytest.mark.parametrize("in_f,out_f", [(65, 65), (32, 65), (128, 128)])
def test_widths_above_64_fail_loudly(in_f, out_f):
    model = make_model(in_f, out_f, 2).to(DEV).set_precision("fp16")
    x1, _ = ragged_pair()
    with torch.no_grad(), pytest.raises(L.FgnnError, match="64"):
        model.node_embedder.forward_fused(x1)
    with pytest.raises(L.FgnnError, match="64"):
        model.node_embedder.forward_fused_train(x1)
