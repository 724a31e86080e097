"""Graphs of up to 4096 vertices through the 16-bit inference path: tensor-core embedder (features- and adjacency-fed,
dense and ragged, both constant_n settings), fused head, device linear assignment and device generators, plus the limits
that stay (N > 4096, 16-bit training above 1024, linear assignment beyond the device's shared memory)."""
import re

import numpy as np
import pytest
import torch

import graph_neural_net_b200 as pkg
from graph_neural_net_b200 import _lib as L, _ops
from graph_neural_net_b200.maskedtensors import maskedtensor as mt
from oracle import fgnn_oracle as O
from tests.helpers import rel_fro

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")


def make_model(c, num_blocks, depth, gen, constant_n=True, randomize_gn=False):
    sd = O.xavier_state_dict(2, c, num_blocks, depth, gen, randomize_gn=randomize_gn)
    node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=num_blocks,
                    in_features=c, out_features=c, depth_of_mlp=depth, constant_n_vertices=constant_n)
    model = pkg.models.Siamese_Node_Exp(2, node_emb)
    model.load_state_dict(sd)
    return model.to(DEV), sd


def device_pairs(generator, G, n, p, seed, sizes=None):
    n_dev = torch.tensor(sizes, dtype=torch.int32, device=DEV) if sizes else None
    return _ops.generate_pairs({"ErdosRenyi": 0, "Regular": 1}[generator], G, n, p, 0.1, seed, n_dev, DEV)


def test_embedder_vs_oracle_above_1024():
    """A ragged batch of n = 1025 and 2049 (C = 32, 3 blocks) against the CPU oracle graph by graph, with the inputs and
    weights of the cfg4-like n <= 1000 test (ER p = 0.2, xavier init): fp16 within 2e-2, bf16 printed (random-init
    weights, DESIGN.md "Precision")."""
    gen = torch.Generator().manual_seed(1025)
    sizes = [1025, 2049]
    model, sd = make_model(32, 3, 3, gen, constant_n=False)
    graphs = [O.synthetic_pair(s, 0.2, 0.1, gen)[0] for s in sizes]
    x = mt.from_list(graphs, dims=(1, 2)).to(DEV)
    with torch.no_grad():
        e = {prec: model.node_embedder.forward_fused(x, prec).tensor.rename(None).cpu() for prec in ("fp16", "bf16")}
        refs = O.node_embedding_ragged(graphs, sd)
    errs = {(s, prec): rel_fro(e[prec][i, :, :s], refs[i]) for i, s in enumerate(sizes) for prec in ("fp16", "bf16")}
    for (s, prec), err in errs.items():
        print(f"PARITY large n={s} {prec}: vs oracle rel err {err:.3e}")
    for i, s in enumerate(sizes):
        assert float(e["fp16"][i, :, s:].abs().sum()) == 0 and float(e["bf16"][i, :, s:].abs().sum()) == 0
        assert errs[(s, "fp16")] < 2e-2


@pytest.mark.parametrize("constant_n", [False, True])
def test_ragged_batch_across_the_old_limit(constant_n, monkeypatch):
    """A ragged fp16 batch padded to 4096: every graph equals the same graph embedded alone (padded to the same N, so
    that constant_n normalises alike), padding is exactly zero, and a run cut into one graph per pass agrees."""
    gen = torch.Generator().manual_seed(4096 + constant_n)
    sizes = [40, 1024, 1025, 2048, 2049, 4096]
    N = max(sizes)
    model, _ = make_model(32, 3, 3, gen, constant_n=constant_n)
    a1, _ = device_pairs("ErdosRenyi", len(sizes), N, 0.05, 31 + constant_n, sizes)
    from graph_neural_net_b200.loaders.data_generator import adjacency_batch_to_tensor_representation
    x = adjacency_batch_to_tensor_representation(a1)
    n_dev = torch.tensor(sizes, dtype=torch.int32, device=DEV)
    keep = []
    params = model.node_embedder._embed_params(keep)
    emb = lambda inp, n: _ops.embed_fwd(params, L.PRECISIONS["fp16"], inp, 32, n)
    with torch.no_grad():
        e = emb(x, n_dev).cpu()
        monkeypatch.setenv("FGNN_TC_WS_GB", "1")           # 5.8 GB per graph: one graph per pass instead of two
        e_passes = emb(x, n_dev).cpu()
        monkeypatch.delenv("FGNN_TC_WS_GB")
        solos = [emb(x[i:i + 1], n_dev[i:i + 1]).cpu()[0] for i in range(len(sizes))]
    assert torch.isfinite(e).all()
    for i, s in enumerate(sizes):
        err_solo = rel_fro(solos[i][:, :s], e[i, :, :s])
        err_pass = rel_fro(e_passes[i, :, :s], e[i, :, :s])
        print(f"PARITY ragged-4096 constant_n={constant_n} n={s}: alone {err_solo:.3e}, one graph per pass {err_pass:.3e}")
        assert err_solo < 5e-3 and err_pass < 5e-3
        assert float(e[i, :, s:].abs().sum()) == 0 and float(e_passes[i, :, s:].abs().sum()) == 0


def test_permutation_equivariance_and_fp32_mode_at_4096():
    """C = 64 at n = 4096, where the CPU oracle is too slow: relabelling the vertices permutes the fp16 embeddings
    (<= 5e-3), and fp16 agrees with the fp32 mode on one pair with a small model (<= 2e-2)."""
    from graph_neural_net_b200.loaders.data_generator import adjacency_batch_to_tensor_representation
    gen = torch.Generator().manual_seed(64)
    n = 4096
    model, _ = make_model(64, 4, 3, gen)
    model.set_precision("fp16")
    a1, a2 = device_pairs("Regular", 1, n, 0.01, 77)
    perm = torch.randperm(n, generator=gen).to(DEV)
    a1p = a1[:, perm][:, :, perm]
    with torch.no_grad():
        e = model.embed({"input": adjacency_batch_to_tensor_representation(a1)})
        ep = model.embed({"input": adjacency_batch_to_tensor_representation(a1p)})
    err_perm = rel_fro(ep.cpu(), e[:, :, perm].cpu())
    print(f"PARITY n=4096 C=64 fp16: permutation equivariance {err_perm:.3e}")
    assert err_perm < 5e-3
    del e, ep
    small, _ = make_model(64, 2, 2, gen)
    out = {}
    with torch.no_grad():
        for prec in ("fp16", "fp32"):
            small.set_precision(prec)
            out[prec] = [small.embed({"input": adjacency_batch_to_tensor_representation(a)}).cpu() for a in (a1, a2)]
            torch.cuda.empty_cache()
    errs = [rel_fro(out["fp16"][k], out["fp32"][k]) for k in range(2)]
    print(f"PARITY n=4096 C=64 fp16 vs fp32 mode (2 blocks, depth 2): {errs[0]:.3e} {errs[1]:.3e}")
    assert max(errs) < 2e-2


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
def test_adjacency_fed_equals_features_fed_at_3000(prec):
    gen = torch.Generator().manual_seed(3000)
    sizes = [3000, 2100]
    N = max(sizes)
    model, _ = make_model(32, 3, 3, gen, constant_n=False)
    adj = torch.zeros((len(sizes), N, N), dtype=torch.uint8)
    graphs = []
    for g, n in enumerate(sizes):
        W = torch.triu(torch.rand((n, n), generator=gen) < 0.05, 1)
        W = W | W.T
        adj[g, :n, :n] = W.to(torch.uint8)
        graphs.append(O.adjacency_to_features(W.float()))
    n_dev = torch.tensor(sizes, dtype=torch.int32, device=DEV)
    with torch.no_grad():
        ref = model.node_embedder.forward_fused(mt.from_list(graphs, dims=(1, 2)).to(DEV), prec).tensor.rename(None)
        out = model.node_embedder.forward_fused_adjacency(adj.to(DEV), prec, n_dev)
    err = rel_fro(out.cpu(), ref.cpu())
    print(f"PARITY n=3000 {prec}: adjacency-fed vs features-fed {err:.3e}")
    assert err < 1e-3
    for g, n in enumerate(sizes):
        assert float(out[g, :, n:].abs().sum()) == 0


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("shape", [(1, 64, 4096, None), (2, 64, 4096, [4096, 2049])])
def test_fused_head_at_4096(prec, shape):
    G, Cc, N, sizes = shape
    gen = torch.Generator().manual_seed(N + G)
    e1 = torch.randn((G, Cc, N), generator=gen)
    e2 = 0.7 * e1 + 0.5 * torch.randn((G, Cc, N), generator=gen)
    n_dev = None
    if sizes is not None:
        n_dev = torch.tensor(sizes, dtype=torch.int32, device=DEV)
        for g, n in enumerate(sizes):
            e1[g, :, n:] = 0
            e2[g, :, n:] = 0
    ce, correct, scores = _ops.head_fused(e1.to(DEV), e2.to(DEV), n_dev, prec, want_scores=True)
    ce2, correct2, _ = _ops.head_fused(e1.to(DEV), e2.to(DEV), n_dev, prec, want_scores=False)
    assert torch.equal(ce, ce2) and torch.equal(correct, correct2)
    for g in range(G):
        n = N if sizes is None else sizes[g]
        ref = e1[g, :, :n].double().t() @ e2[g, :, :n].double()
        got = scores[g].cpu().double()
        assert float((got[:n, :n] - ref).norm() / ref.norm()) < 1e-5
        if n < N:
            assert float(got[n:, :].abs().max()) == 0.0 and float(got[:, n:].abs().max()) == 0.0
        ref_ce = float(torch.nn.functional.cross_entropy(ref, torch.arange(n), reduction="sum"))
        assert abs(float(ce[g]) - ref_ce) < 1e-4 * max(1.0, abs(ref_ce)), (g, float(ce[g]), ref_ce)
        assert int(correct[g]) == int((ref.argmax(1) == torch.arange(n)).sum())


@pytest.mark.parametrize("n,sizes", [(3900, None), (4096, [4096, 3900])])
def test_linear_assignment_equals_scipy_at_large_n(n, sizes):
    from scipy.optimize import linear_sum_assignment
    from graph_neural_net_b200.toolbox.metrics import linear_assignment
    gen = torch.Generator().manual_seed(n)
    G = len(sizes) if sizes else 1
    scores = torch.randn((G, n, n), generator=gen) * 3
    scores[0] += 4 * torch.eye(n)
    x = scores.to(DEV)
    if sizes:
        x = mt.from_list([scores[i, :s, :s] for i, s in enumerate(sizes)], dims=(0, 1)).to(DEV)
    cols, correct, cost = linear_assignment(x)
    cols, correct, cost = cols.cpu().numpy(), correct.cpu().numpy(), cost.cpu().numpy()
    for g in range(G):
        m = sizes[g] if sizes else n
        ref_cost_mat = -torch.log_softmax(scores[g, :m, :m], -1).numpy().astype(np.float64)
        rows, preds = linear_sum_assignment(ref_cost_mat)
        assert np.array_equal(cols[g, :m], preds), g
        assert np.all(cols[g, m:] == -1)
        assert correct[g] == int(np.sum(preds == np.arange(m)))
        assert abs(cost[g] - ref_cost_mat[rows, preds].sum()) < 1e-5 * max(1.0, abs(cost[g]))


@pytest.mark.parametrize("n", [2048, 4096])
def test_generators_at_large_n(n):
    """Regular: every vertex of degree exactly d, symmetric, no loops (bitmap in the workspace above N = 1264).
    ErdosRenyi: density within 4 sigma.  The same seed gives the same bytes."""
    p = 0.01
    r1, _ = device_pairs("Regular", 2, n, p, 5, [n, n - 3])
    r1b, _ = device_pairs("Regular", 2, n, p, 5, [n, n - 3])
    assert torch.equal(r1, r1b)
    for g, m in enumerate([n, n - 3]):
        d = int(p * m) + ((m * int(p * m)) & 1)
        a = r1[g, :m, :m].long()
        assert torch.equal(a, a.T) and int(a.diagonal().sum()) == 0
        assert bool((a.sum(1) == d).all()), (m, d)
        assert int(r1[g].sum()) == int(a.sum())
    e1, e2 = device_pairs("ErdosRenyi", 1, n, 0.05, 9)
    e1b, e2b = device_pairs("ErdosRenyi", 1, n, 0.05, 9)
    assert torch.equal(e1, e1b) and torch.equal(e2, e2b)
    a = e1[0].long()
    assert torch.equal(a, a.T) and int(a.diagonal().sum()) == 0
    pairs = n * (n - 1) // 2
    edges = int(a.sum()) // 2
    assert abs(edges - 0.05 * pairs) < 4 * (pairs * 0.05 * 0.95) ** 0.5


def _limit_in(msg, limit):
    return str(limit) in re.findall(r"\d+", msg)


def test_limits_fail_loudly():
    gen = torch.Generator().manual_seed(1)
    model, _ = make_model(32, 2, 2, gen)
    x = torch.zeros((1, 2, 4097, 4097), device=DEV)
    with torch.no_grad(), pytest.raises(L.FgnnError) as ei:
        model.node_embedder.forward_fused(x, "fp16")
    assert _limit_in(str(ei.value), 4096)
    del x
    e = torch.zeros((1, 32, 4097), device=DEV)
    with pytest.raises(L.FgnnError) as ei:
        _ops.head_fused(e, e, None, "fp16")
    assert _limit_in(str(ei.value), 4096)
    with pytest.raises(L.FgnnError) as ei:
        device_pairs("ErdosRenyi", 1, 4097, 0.05, 1)
    assert _limit_in(str(ei.value), 4096)
    # 16-bit training stops at 1024
    model.set_precision("fp16")
    x = torch.zeros((1, 2, 1025, 1025), device=DEV)
    with pytest.raises(L.FgnnError) as ei:
        model.embed({"input": x})
    assert _limit_in(str(ei.value), 1024)
    # linear assignment: the limit the message states is where it stops
    from graph_neural_net_b200.toolbox.metrics import linear_assignment
    with pytest.raises(L.FgnnError) as ei:
        linear_assignment(torch.zeros((1, 6000, 6000), device=DEV))
    limit = int(re.search(r"N <= (\d+)", str(ei.value)).group(1))
    assert limit >= 4096
    with pytest.raises(L.FgnnError) as ei:
        linear_assignment(torch.zeros((1, limit + 1, limit + 1), device=DEV))
    assert _limit_in(str(ei.value), limit)
