"""GPU tests of graph pairs whose two graphs differ in size (n1 != n2, padded to N1 != N2): the tensor-core head forward
and backward, the CUDA-core scores and cross-entropy, the rectangular device LAP, and the model end to end.  The oracle
is a float64 loop per graph: s = e1[:, :n1]^T e2[:, :n2], the cross-entropy and arg-max of rows with a target
(i < n2), and scipy's linear_sum_assignment on -log_softmax(s)."""
import numpy as np
import pytest
import torch
from scipy.optimize import linear_sum_assignment

import graph_neural_net_b200 as pkg
from graph_neural_net_b200 import _lib as L
from graph_neural_net_b200 import _ops
from graph_neural_net_b200.loaders.loaders import collate_fn_pair
from graph_neural_net_b200.maskedtensors import maskedtensor as mt
from graph_neural_net_b200.toolbox.losses import triplet_loss
from graph_neural_net_b200.toolbox.metrics import accuracy_linear_assignment, accuracy_max, linear_assignment
from graph_neural_net_b200.training import FlatAdam, train_step_flat
from oracle import fgnn_oracle as O
from tests.helpers import load_golden, rel_fro, state_dict_of

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# (N1, N2, n1 or None, n2 or None): dense shapes and one ragged batch padded differently on the two sides
SHAPES = [(50, 80, None, None), (200, 129, None, None), (300, 520, None, None), (1000, 4096, None, None),
          (100, 300, [100, 37, 64], [250, 300, 65])]


def make_pair(N1, N2, n1, n2, C=32, seed=0):
    """e1[:, i] ~ e2[:, i] + noise for i < min(n1, n2): the scores peak near the diagonal.  Padding holds garbage."""
    gen = torch.Generator().manual_seed(seed)
    G = len(n1) if n1 else 2
    n1 = n1 or [N1] * G
    n2 = n2 or [N2] * G
    e2 = torch.randn(G, C, N2, generator=gen) * (4.0 / C) ** 0.5
    e1 = torch.randn(G, C, N1, generator=gen) * (4.0 / C) ** 0.5
    m = min(N1, N2)
    e1[:, :, :m] = e2[:, :, :m] + 0.5 * e1[:, :, :m]
    return e1, e2, n1, n2


def oracle(e1, e2, n1, n2):
    """Per graph: fp64 scores (N1, N2) zero outside n1 x n2, ce_sum and #correct over rows i < min(n1, n2)."""
    G, _, N1 = e1.shape
    N2 = e2.shape[2]
    S = torch.zeros(G, N1, N2, dtype=torch.float64)
    ce, ok, arg = [], [], torch.full((G, N1), -1, dtype=torch.int64)
    for g in range(G):
        s = e1[g, :, :n1[g]].double().T @ e2[g, :, :n2[g]].double()
        S[g, :n1[g], :n2[g]] = s
        r = min(n1[g], n2[g])
        lse = torch.logsumexp(s, dim=1)
        ce.append(float((lse[:r] - s.diagonal()[:r]).sum()))
        am = s.argmax(dim=1)
        arg[g, :n1[g]] = am
        ok.append(int((am[:r] == torch.arange(r)).sum()))
    return S, np.array(ce), np.array(ok)


def sizes_dev(n):
    return torch.tensor(n, dtype=torch.int32, device=DEV)


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("N1,N2,n1,n2", SHAPES)
def test_head_forward_two_sizes(N1, N2, n1, n2, prec):
    e1, e2, n1, n2 = make_pair(N1, N2, n1, n2, seed=N1 + N2)
    S, ce_ref, ok_ref = oracle(e1, e2, n1, n2)
    a, b, d1, d2 = e1.to(DEV), e2.to(DEV), sizes_dev(n1), sizes_dev(n2)
    ce, ok, s = _ops.head_fused(a, b, d1, prec, want_scores=True, n2_dev=d2)
    assert s.shape == (len(n1), N1, N2)
    err = rel_fro(s.cpu(), S)
    print(f"head {prec} N1={N1} N2={N2}: scores rel err {err:.2e}")
    assert err <= 1e-5
    assert np.allclose(ce.cpu().numpy(), ce_ref, rtol=1e-5, atol=1e-3)
    assert (ok.cpu().numpy() == ok_ref).all()
    # the training forward is the inference head bit for bit
    ce_t, ok_t = _ops.HeadFunction.apply(a, b, d1, prec, d2)
    assert torch.equal(ce_t, ce) and torch.equal(ok_t, ok)


def fp64_grads(e1, e2, coef, n1, n2):
    a = e1.double().clone().requires_grad_(True)
    b = e2.double().clone().requires_grad_(True)
    total = 0.0
    for g in range(e1.shape[0]):
        s = a[g, :, :n1[g]].T @ b[g, :, :n2[g]]
        r = min(n1[g], n2[g])
        total = total + coef[g].double() * (torch.logsumexp(s[:r], dim=1) - s.diagonal()[:r]).sum()
    total.backward()
    return a.grad, b.grad


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("N1,N2,n1,n2", SHAPES)
def test_head_backward_two_sizes(N1, N2, n1, n2, prec):
    e1, e2, n1, n2 = make_pair(N1, N2, n1, n2, seed=3 * N1 + N2)
    coef = torch.rand(len(n1)) + 0.25
    r1, r2 = fp64_grads(e1, e2, coef, n1, n2)
    d1, d2 = sizes_dev(n1), sizes_dev(n2)
    runs = []
    for _ in range(2):
        x1, x2 = e1.to(DEV).requires_grad_(True), e2.to(DEV).requires_grad_(True)
        ce, _ = _ops.HeadFunction.apply(x1, x2, d1, prec, d2)
        ce.backward(coef.to(DEV))
        runs.append((x1.grad.clone(), x2.grad.clone()))
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])     # deterministic
    g1, g2 = runs[0]
    for gr, n in ((g1, n1), (g2, n2)):
        assert torch.isfinite(gr).all()
        for k, nk in enumerate(n):
            assert torch.count_nonzero(gr[k, :, nk:]) == 0
    # the CUDA-core pair path
    y1, y2 = e1.to(DEV).requires_grad_(True), e2.to(DEV).requires_grad_(True)
    ce_ref, _ = _ops.CrossEntropyIdentityFunction.apply(_ops.ScoresFunction.apply(y1, y2, d1, d2), d1, d2)
    ce_ref.backward(coef.to(DEV))
    e = [rel_fro(g1.cpu(), r1), rel_fro(g2.cpu(), r2), rel_fro(g1, y1.grad), rel_fro(g2, y2.grad)]
    print(f"head bwd {prec} N1={N1} N2={N2}: vs fp64 {e[0]:.2e} {e[1]:.2e}; vs CUDA-core {e[2]:.2e} {e[3]:.2e}")
    assert max(e) <= 1e-4
    assert rel_fro(y1.grad.cpu(), r1) <= 1e-5 and rel_fro(y2.grad.cpu(), r2) <= 1e-5


@pytest.mark.parametrize("N1,N2,n1,n2", SHAPES[:3] + SHAPES[4:])
def test_fp32_scores_and_ce_two_sizes(N1, N2, n1, n2):
    e1, e2, n1, n2 = make_pair(N1, N2, n1, n2, seed=N1 * 7 + N2)
    S, ce_ref, ok_ref = oracle(e1, e2, n1, n2)
    d1, d2 = sizes_dev(n1), sizes_dev(n2)
    s = _ops.ScoresFunction.apply(e1.to(DEV), e2.to(DEV), d1, d2)
    assert rel_fro(s.cpu(), S) <= 1e-5
    ce, ok, _, arg = _ops.ce_argmax(s, d1, d2, want_argmax=True)
    assert np.allclose(ce.cpu().numpy(), ce_ref, rtol=1e-5, atol=1e-3)
    assert (ok.cpu().numpy() == ok_ref).all()
    arg_ref = torch.full(arg.shape, -1, dtype=torch.int32)
    for g in range(len(n1)):
        arg_ref[g, :n1[g]] = S[g, :n1[g], :n2[g]].argmax(dim=1).to(torch.int32)
    assert torch.equal(arg.cpu(), arg_ref)


def scipy_lap(S, n1, n2):
    cols = np.full((S.shape[0], S.shape[1]), -1)
    cost = []
    for g in range(S.shape[0]):
        c = -torch.log_softmax(S[g, :n1[g], :n2[g]].float(), -1).numpy()
        r, k = linear_sum_assignment(c)
        cols[g, r] = k
        cost.append(c[r, k].astype(np.float64).sum())
    return cols, np.array(cost)


@pytest.mark.parametrize("seed,case", enumerate(["n1<n2", "n1>n2", "ragged", "ties-n1<n2", "ties-n1>n2"]))
def test_lap_two_sizes_equals_scipy(seed, case):
    gen = torch.Generator().manual_seed(100 + seed)
    N1, N2, n1, n2 = {"n1<n2": (40, 70, [40, 40], [70, 70]), "n1>n2": (90, 33, [90, 90], [33, 33]),
                      "ragged": (60, 50, [60, 12, 30, 1], [50, 40, 7, 50]),
                      "ties-n1<n2": (30, 45, [30, 30], [45, 45]), "ties-n1>n2": (45, 30, [45, 20], [30, 30])}[case]
    if case.startswith("ties"):
        S = torch.randint(0, 3, (len(n1), N1, N2), generator=gen).float()
    else:
        S = torch.randn(len(n1), N1, N2, generator=gen) * 3
    for g in range(len(n1)):
        S[g, n1[g]:], S[g, :, n2[g]:] = 0, 0
    if n1 == [N1] * len(n1) and n2 == [N2] * len(n2):
        x = S.to(DEV)
    else:
        x = mt.from_list([S[g, :n1[g], :n2[g]] for g in range(len(n1))], dims=(0, 1)).to(DEV)
    cols, correct, cost = linear_assignment(x)
    ref_cols, ref_cost = scipy_lap(S, n1, n2)
    assert (cols.cpu().numpy() == ref_cols).all()
    # the kernel forms the log-softmax constants with the device's expf / logf: costs agree to fp32 rounding
    assert np.allclose(cost.cpu().numpy(), ref_cost, rtol=1e-5, atol=1e-4)
    hits = [int((ref_cols[g, :n1[g]] == np.arange(n1[g])).sum()) for g in range(len(n1))]
    assert correct.cpu().tolist() == hits


def test_head_refuses_more_than_4096_columns():
    e = torch.zeros(1, 32, 64, device=DEV)
    with pytest.raises(L.FgnnError, match="4096"):
        _ops.head_fused(e, torch.zeros(1, 32, 4097, device=DEV), None, "fp16")


# ---- end to end: graph 2 = noisy copy of graph 1 plus appended random vertices --------------------------------------
def grown_pair(n1, n2, gen, p=0.2, noise=0.05):
    """Graph 2 holds a noisy copy of graph 1 on its first n1 vertices, so row i <-> column i is the ground truth."""
    W1, W1n = O.synthetic_pair(n1, p, noise, gen)
    W2 = (torch.rand(n2, n2, generator=gen) < p).float().triu(1)
    W2 = W2 + W2.T
    m = min(n1, n2)
    W2[:m, :m] = W1n[0][:m, :m]
    return W1[0], W2


def setup_model(c=32, nb=3, seed=5):
    gen = torch.Generator().manual_seed(seed)
    sd = O.xavier_state_dict(2, c, nb, 3, gen, randomize_gn=True)
    node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=nb,
                    in_features=c, out_features=c, depth_of_mlp=3)

    def make():
        m = pkg.models.Siamese_Node_Exp(2, dict(node_emb))
        m.load_state_dict(sd)
        return m.to(DEV)
    return sd, make


SIZES = [(30, 45), (50, 50), (20, 64), (41, 41 + 17)]


def batch_of(sizes, seed=11):
    gen = torch.Generator().manual_seed(seed)
    pairs = [grown_pair(a, b, gen) for a, b in sizes]
    feats = [(O.adjacency_to_features(w1), O.adjacency_to_features(w2)) for w1, w2 in pairs]
    m1, m2 = collate_fn_pair(feats)
    return feats, {"input": m1.to(DEV)}, {"input": m2.to(DEV)}


def test_end_to_end_fp32_and_fp16():
    sd, make = setup_model()
    feats, x1, x2 = batch_of(SIZES)
    sd64 = {k: v.double() for k, v in sd.items()}
    # GraphNorm's n is each side's padded size (constant_n_vertices=True, the reference's default)
    N1, N2 = max(a for a, _ in SIZES), max(b for _, b in SIZES)
    emb = lambda f, n: O.node_embedding(f[None].double(), sd64, n=float(n))[0]  # noqa: E731
    ref = [emb(a, N1).T @ emb(b, N2) for a, b in feats]
    model = make()
    with torch.no_grad():
        s = model(x1, x2)
        e1, e2 = model.embed(x1), model.embed(x2)
    for g, (a, b) in enumerate(feats):
        n1, n2 = a.shape[-1], b.shape[-1]
        for e, f, n in ((e1, a, N1), (e2, b, N2)):
            assert rel_fro(e.tensor.rename(None)[g, :, :f.shape[-1]].cpu(), emb(f, n)) <= 1e-4
        sg = s.tensor.rename(None)[g].cpu()
        assert rel_fro(sg[:n1, :n2], ref[g]) <= 1e-4
        assert torch.count_nonzero(sg[n1:]) == 0 and torch.count_nonzero(sg[:, n2:]) == 0
    loss_ref = float(O.triplet_loss(ref))
    loss = float(triplet_loss()(s))
    assert abs(loss - loss_ref) <= 1e-4 * max(1.0, abs(loss_ref))
    assert accuracy_max(s) == O.accuracy_max(ref)
    assert accuracy_linear_assignment(s) == O.accuracy_linear_assignment(ref)
    l32, ok32, rows32 = model.loss_and_accuracy(x1, x2)
    assert int(rows32) == sum(a for a, _ in SIZES) and abs(float(l32) - loss_ref) <= 1e-4 * max(1.0, abs(loss_ref))
    model.set_precision("fp16")
    with torch.no_grad():
        s16 = model(x1, x2)
    l16, ok16, rows16 = model.loss_and_accuracy(x1, x2)
    err = rel_fro(s16.tensor.rename(None).cpu(), s.tensor.rename(None).cpu())
    print(f"end to end: fp32 loss {loss:.6f} (oracle {loss_ref:.6f}); fp16 scores rel err {err:.2e} loss {float(l16):.6f}")
    assert err <= 5e-3 and abs(float(l16) - loss_ref) <= 2e-2 and int(rows16) == int(rows32)
    # dense inputs of different padded sizes
    with torch.no_grad():
        d = model({"input": feats[0][0][None].to(DEV)}, {"input": feats[0][1][None].to(DEV)})
    assert d.shape == (1, SIZES[0][0], SIZES[0][1])


def test_loss_refuses_n1_above_n2_end_to_end():
    _, make = setup_model()
    _, x1, x2 = batch_of([(30, 20), (20, 30)])
    model = make()
    with pytest.raises(ValueError, match="n1=30 > n2=20"):
        triplet_loss()(model(x1, x2))
    # scores and the assignment are defined for any sizes
    with torch.no_grad():
        s = model(x1, x2)
    cols, _, _ = linear_assignment(s)
    assert (cols[0, :30] >= 0).sum() == 20 and (cols[1, :20] >= 0).all()


@pytest.mark.parametrize("fused_head", [False, True])
def test_train_step_two_sizes(fused_head):
    _, make = setup_model()
    _, x1, x2 = batch_of(SIZES)
    ref = make()
    ref_loss = train_step_flat(ref, FlatAdam(ref.parameters(), lr=ref.lr), x1, x2)[0]
    _ops.GradScale.log2, _ops.GradScale._good = 9, 0
    model = make().set_precision("fp16")
    opt = FlatAdam(model.parameters(), lr=model.lr)
    losses, rows = [], set()
    for _ in range(6):
        loss, _, n = train_step_flat(model, opt, x1, x2, fused_head=fused_head)
        losses.append(loss)
        rows.add(n)
    print(f"train_step_flat fused_head={fused_head}: fp32 {ref_loss:.5f}, fp16 {[round(v, 4) for v in losses]}")
    assert abs(losses[0] - ref_loss) <= 5e-3 and losses[-1] < losses[0]
    assert rows == {sum(a for a, _ in SIZES)}


def test_labels_on_trained_model():
    """Permuting graph 2 by pi and passing pi as the labels gives the identity accuracies of the unpermuted pairs."""
    z = load_golden("trained_er50_c32")
    n, c, nb, depth, _ = [int(v) for v in z["meta"]]
    node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=nb,
                    in_features=c, out_features=c, depth_of_mlp=depth)
    model = pkg.models.Siamese_Node_Exp(2, node_emb)
    model.load_state_dict(state_dict_of(z))
    model = model.to(DEV)
    f = lambda W: torch.stack([O.adjacency_to_features(torch.from_numpy(w.astype(np.float32))) for w in W]).to(DEV)  # noqa: E731
    gen = torch.Generator().manual_seed(17)
    perms = [torch.randperm(n, generator=gen) for _ in range(z["W2"].shape[0])]
    W2p = np.stack([w[p][:, p] for w, p in zip(z["W2"], [p.numpy() for p in perms])])
    # graph 2's vertex p[k] is the old vertex k... so row i's match is the position of i in p
    labels = [torch.argsort(p).numpy() for p in perms]
    with torch.no_grad():
        s = model({"input": f(z["W1"])}, {"input": f(z["W2"])})
        sp = model({"input": f(z["W1"])}, {"input": f(W2p)})
    assert accuracy_max(sp, labels=labels) == accuracy_max(s)
    assert accuracy_linear_assignment(sp, labels=labels) == accuracy_linear_assignment(s)
    assert accuracy_max(sp, labels=labels, aggregate_score=False) == accuracy_max(s, aggregate_score=False)


def test_equal_size_batches_unchanged():
    """An equal-size ragged batch gives what the single-size call (graph 1's sizes for both sides) gives."""
    _, make = setup_model()
    _, x1, x2 = batch_of([(30, 30), (50, 50), (17, 17)])
    model = make()
    for prec in ("fp32", "fp16"):
        model.set_precision(prec)
        with torch.no_grad():
            s = model(x1, x2)
            e1, e2 = model.embed(x1), model.embed(x2)
            t1, t2, d = e1.tensor.rename(None), e2.tensor.rename(None), e1.sizes_i32()
            old = (_ops.ScoresFunction.apply(t1, t2, d) if prec == "fp32"
                   else _ops.head_fused(t1, t2, d, prec, want_scores=True)[2])
        assert torch.equal(s.tensor.rename(None), old)
        assert s.sizes_host("N") == s.sizes_host("N_") == [30, 50, 17]
