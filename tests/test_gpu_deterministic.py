"""GPU tests of the deterministic mode: with torch.use_deterministic_algorithms(True) (or FGNN_DETERMINISTIC=1) the
library sums every cross-CTA partial in a fixed order, so two runs from identically seeded models give bit-identical
embeddings, losses, gradients and optimiser states.  The deterministic results also agree with the default mode's
within the spread the other tests allow, and pass the golden / oracle comparisons of test_gpu_tc_train.py."""
import pytest
import torch

import graph_neural_net_b200 as pkg
from graph_neural_net_b200 import _ops
from graph_neural_net_b200.maskedtensors import maskedtensor as mt
from graph_neural_net_b200.training import FlatAdam, train_step, train_step_flat
from oracle import fgnn_oracle as O
from tests import test_gpu_tc_train as T
from tests.helpers import rel_fro
from tests.test_gpu_pair_sizes import SIZES, batch_of

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture
def deterministic():
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=warn)


def node_emb(c, nb=4, depth=3):
    return dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=nb, in_features=c,
                out_features=c, depth_of_mlp=depth)


def make_model(c, precision, seed=3787, nb=4):
    gen = torch.Generator().manual_seed(seed)
    m = pkg.models.Siamese_Node_Exp(2, node_emb(c, nb))
    m.load_state_dict(O.xavier_state_dict(2, c, nb, 3, gen, randomize_gn=True))
    return m.to(DEV).set_precision(precision)


def pairs(sizes, seed=5):
    gen = torch.Generator().manual_seed(seed)
    return [O.synthetic_pair(s, 0.2, 0.1, gen) for s in sizes]


def dense(n, G, seed=5):
    ps = pairs([n] * G, seed)
    return {"input": torch.stack([p[0] for p in ps]).to(DEV)}, {"input": torch.stack([p[1] for p in ps]).to(DEV)}


def ragged(sizes, seed=5):
    ps = pairs(sizes, seed)
    return ({"input": mt.from_list([p[0] for p in ps], dims=(1, 2)).to(DEV)},
            {"input": mt.from_list([p[1] for p in ps], dims=(1, 2)).to(DEV)})


def flat_run(c, precision, x1, x2, steps=3, fused_head=False):
    """steps of train_step_flat from a fresh model: (losses, corrects, flat_p, flat_m, flat_v)."""
    _ops.GradScale.log2, _ops.GradScale._good = 9, 0
    model = make_model(c, precision)
    opt = FlatAdam(model.parameters(), lr=model.lr)
    out = [train_step_flat(model, opt, x1, x2, fused_head=fused_head) for _ in range(steps)]
    torch.cuda.synchronize()
    return [o[0] for o in out], [o[1:] for o in out], opt.flat_p.clone(), opt.flat_m.clone(), opt.flat_v.clone()


def assert_identical(a, b, label):
    la, ca, *ta = a
    lb, cb, *tb = b
    assert la == lb and ca == cb, (label, la, lb, ca, cb)
    for u, v, name in zip(ta, tb, ("flat_p", "flat_m", "flat_v")):
        assert torch.equal(u, v), (label, name, float((u - v).abs().max()))
    print(f"DETERMINISTIC {label}: losses {[round(v, 6) for v in la]} bit-identical over two runs")


@pytest.mark.parametrize("fused_head", [False, True])
@pytest.mark.parametrize("prec", ["fp16", "bf16"])
def test_train_step_flat_bit_identical(prec, fused_head, deterministic):
    x1, x2 = dense(50, 16)
    assert_identical(flat_run(32, prec, x1, x2, fused_head=fused_head), flat_run(32, prec, x1, x2, fused_head=fused_head),
                     f"ER n=50 x16 {prec} fused_head={fused_head}")


def test_ragged_recompute_plan_bit_identical(deterministic, monkeypatch):
    monkeypatch.setenv("FGNN_TC_TRAIN_WS_GB", "0")
    monkeypatch.setenv("FGNN_TC_CHUNK", "3")
    x1, x2 = ragged([50, 23, 37, 64, 130, 41, 77])
    assert_identical(flat_run(32, "fp16", x1, x2), flat_run(32, "fp16", x1, x2), "ragged recompute chunk=3")


@pytest.mark.parametrize("fused_head", [False, True])
def test_unequal_pair_sizes_bit_identical(fused_head, deterministic):
    _, x1, x2 = batch_of(SIZES)
    assert_identical(flat_run(32, "fp16", x1, x2, fused_head=fused_head),
                     flat_run(32, "fp16", x1, x2, fused_head=fused_head), f"unequal sizes fused_head={fused_head}")


def test_fp32_train_step_bit_identical(deterministic):
    x1, x2 = dense(30, 6)

    def run():
        model = make_model(16, "fp32", nb=2)
        opt = model.configure_optimizers()["optimizer"]
        res = [train_step(model, opt, x1, x2) for _ in range(2)]
        grads = [p.grad.clone() for p in model.parameters()]
        return res, [p.detach().clone() for p in model.parameters()], grads

    (ra, pa, ga), (rb, pb, gb) = run(), run()
    assert ra == rb, (ra, rb)
    for u, v in zip(pa + ga, pb + gb):
        assert torch.equal(u, v), float((u - v).abs().max())


def embed_both(model, x):
    """(default-mode, deterministic-mode) embeddings of the same input."""
    with torch.no_grad():
        e0 = model.embed(x)
        torch.use_deterministic_algorithms(True)
        try:
            e1, e2 = model.embed(x), model.embed(x)
        finally:
            torch.use_deterministic_algorithms(False)
    assert torch.equal(e1, e2)
    return e0, e1


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
def test_inference_bit_identical_and_close_to_default(prec):
    model = make_model(64, prec)
    x1, x2 = dense(500, 4)
    e0, e1 = embed_both(model, x1)
    err = rel_fro(e1.cpu(), e0.cpu())
    print(f"{prec} n=500 C=64: deterministic vs default embeddings {err:.2e}")
    assert err <= 1e-6
    torch.use_deterministic_algorithms(True)
    try:
        a = model.loss_and_accuracy(x1, x2)
        b = model.loss_and_accuracy(x1, x2)
    finally:
        torch.use_deterministic_algorithms(False)
    assert [float(v) for v in a] == [float(v) for v in b]
    big = make_model(32, prec, nb=2)
    xb, _ = dense(2048, 1)
    e0, e1 = embed_both(big, xb)
    err = rel_fro(e1.cpu(), e0.cpu())
    print(f"{prec} N=2048: deterministic vs default embeddings {err:.2e}")
    assert err <= 1e-6


def grads_of(model, x1, x2):
    _ops.GRAD_SINK.clear()
    for p in model.parameters():
        p.grad = None
    loss = T.triplet_loss("mean")(model(x1, x2))
    loss.backward()
    return float(loss.detach()), torch.cat([p.grad.detach().flatten() for p in model.parameters()])


def test_gradients_close_to_default_mode():
    x1, x2 = dense(50, 16)
    model = make_model(32, "fp16")
    _ops.GradScale.log2 = 9
    l0, g0 = grads_of(model, x1, x2)
    torch.use_deterministic_algorithms(True)
    try:
        l1, g1 = grads_of(model, x1, x2)
    finally:
        torch.use_deterministic_algorithms(False)
    err = float((g1 - g0).norm() / g0.norm())
    print(f"deterministic vs default: loss {l1:.7f} / {l0:.7f}, gradients {err:.2e}")
    assert abs(l1 - l0) <= 1e-6 * max(1.0, abs(l0))
    assert err <= 1e-5


def test_backward_keeps_the_forward_mode():
    """Toggling the flag between calls switches the mode; a backward runs in its forward's mode (its workspace and
    plan were chosen for it)."""
    x1, x2 = dense(50, 8)
    model = make_model(32, "fp16")
    _ops.GradScale.log2 = 9
    torch.use_deterministic_algorithms(True)
    try:
        assert _ops.deterministic_bit() == pkg._lib.FGNN_DETERMINISTIC
        _, ref = grads_of(model, x1, x2)
        # forward deterministic, backward after the flag went off: still deterministic, bit for bit
        _ops.GRAD_SINK.clear()
        for p in model.parameters():
            p.grad = None
        loss = T.triplet_loss("mean")(model(x1, x2))
    finally:
        torch.use_deterministic_algorithms(False)
    assert _ops.deterministic_bit() == 0
    loss.backward()
    assert torch.equal(torch.cat([p.grad.detach().flatten() for p in model.parameters()]), ref)
    # forward in the default mode, backward with the flag on: runs (default mode), same gradients up to rounding
    for p in model.parameters():
        p.grad = None
    loss = T.triplet_loss("mean")(model(x1, x2))
    torch.use_deterministic_algorithms(True)
    try:
        loss.backward()
    finally:
        torch.use_deterministic_algorithms(False)
    g = torch.cat([p.grad.detach().flatten() for p in model.parameters()])
    assert float((g - ref).norm() / ref.norm()) <= 1e-5


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("name", ["cfg1_er50_c32", "cfg2_er200_c32"])
def test_golden_and_oracle_gradients_in_deterministic_mode(name, prec, deterministic):
    T.test_tc_training_gradients_match_reference_autograd(name, prec)
