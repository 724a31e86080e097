"""GPU parity tests of the tensor-core path (FGNN_BF16 / FGNN_FP16) through the C ABI.

Oracles: torch fp64 algebra on 16-bit-rounded operands for the isolated kernels, the CPU oracle /
golden vectors of the reference for whole embedders, the fp32 CUDA path at sizes the CPU oracle
cannot reach.  Tolerances: the north_star asks <= 2e-2 relative on node embeddings for the 16-bit
mode.  With fp16 operands (FGNN_FP16, same tcgen05 kind::f16 instruction and speed) that bar is met
and asserted; with bf16 operands the error on random-init networks is 3e-2 .. 2e-1 depending on
n / width -- rounding the weights and hidden activations to 8 mantissa bits is amplified by the
four GraphNorm re-normalisations (DESIGN.md "Precision") -- so bf16 asserts its measured envelope.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import graph_neural_net_b200 as pkg
from graph_neural_net_b200 import _lib as L, _ops
from graph_neural_net_b200.maskedtensors import maskedtensor as mt
from oracle import fgnn_oracle as O
from tests.helpers import load_golden, state_dict_of, rel_fro

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
EMB_TOL = {"fp16": 5e-2, "bf16": 5e-1}      # small graphs (n<=130) are the worst conditioned; n=500 asserts 2e-2 below
TDT = {"bf16": torch.bfloat16, "fp16": torch.float16}


def tc_matmul(prec, a, b, n_dev=None):
    lib = pkg.get_lib()
    G, Cc, N, _ = a.shape
    out = torch.empty_like(a)
    ws = L.workspace(a.device, lib.fgnn_debug_tc_matmul_workspace_bytes(G, Cc, N))
    L.check(lib.fgnn_debug_tc_matmul(L.PRECISIONS[prec], L.ptr(a), L.ptr(b), L.ptr(out), G, Cc, N,
                                     L.ptr(n_dev) if n_dev is not None else None, L.ptr(ws), ws.numel(),
                                     L.stream_ptr(a.device)), "fgnn_debug_tc_matmul")
    return out


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
@pytest.mark.parametrize("shape,sizes", [((2, 3, 40), None), ((1, 2, 64), None), ((2, 2, 100), None),
                                         ((1, 2, 200), None), ((1, 1, 500), None),
                                         ((3, 2, 150), [150, 70, 33]), ((2, 1, 1000), [1000, 257]),
                                         ((3, 2, 300), [300, 129, 40])])
def test_tc_matmul_vs_fp64_on_rounded_operands(prec, shape, sizes):
    G, Cc, N = shape
    gen = torch.Generator().manual_seed(N + G)
    a = torch.randn((G, Cc, N, N), generator=gen).to(DEV)
    b = torch.randn((G, Cc, N, N), generator=gen).to(DEV)
    n_dev = torch.tensor(sizes, dtype=torch.int32, device=DEV) if sizes else None
    out = tc_matmul(prec, a, b, n_dev)
    ar, br = a.to(TDT[prec]).double(), b.to(TDT[prec]).double()
    tol = 2.5e-3 if prec == "bf16" else 4e-4           # one rounding of the output to 8 / 11 bits
    for g in range(G):
        n = sizes[g] if sizes else N
        ref = torch.matmul(ar[g, :, :n, :n], br[g, :, :n, :n])
        assert rel_fro(out[g, :, :n, :n].cpu(), ref.cpu()) < tol
        assert float(out[g, :, n:, :].abs().sum()) == 0 and float(out[g, :, :, n:].abs().sum()) == 0


@pytest.mark.parametrize("prec", ["bf16", "fp16"])
@pytest.mark.parametrize("c_in,c_out,depth,G,N,sizes", [(64, 64, 3, 2, 40, None), (2, 64, 3, 1, 50, None),
                                                        (128, 64, 3, 1, 72, None), (32, 32, 3, 2, 40, None),
                                                        (2, 32, 2, 2, 30, [30, 17]), (34, 32, 3, 1, 50, None),
                                                        (66, 64, 1, 1, 24, None)])
def test_tc_mlp_block_vs_oracle(prec, c_in, c_out, depth, G, N, sizes):
    lib = pkg.get_lib()
    gen = torch.Generator().manual_seed(7 * N + c_out + depth)
    x = torch.randn((G, c_in, N, N), generator=gen)
    ws_ = [torch.randn((c_out, c_in if k == 0 else c_out), generator=gen) / (c_in if k == 0 else c_out) ** 0.5
           for k in range(depth)]
    bs = [torch.randn(c_out, generator=gen) * 0.1 for _ in range(depth)]
    gw = 1 + 0.3 * torch.randn(c_out, generator=gen)
    gb = 0.2 * torch.randn(c_out, generator=gen)
    sd = {"m.gn.weight": gw, "m.gn.bias": gb}
    for k in range(depth):
        sd[f"m.convs.{k}.weight"] = ws_[k].reshape(c_out, -1, 1, 1)
        sd[f"m.convs.{k}.bias"] = bs[k]
    keep = []
    # ragged cases use the per-graph n (constant_n_vertices=False), which is what the per-graph oracle computes
    p = _ops.make_mlp_params([w.to(DEV) for w in ws_], [b.to(DEV) for b in bs], gw.to(DEV), gb.to(DEV), 1e-5, keep,
                             constant_n=sizes is None)
    xd = x.to(DEV)
    n_dev = torch.tensor(sizes, dtype=torch.int32, device=DEV) if sizes else None
    y = torch.empty((G, c_out, N, N), device=DEV)
    wsb = L.workspace(DEV, lib.fgnn_debug_tc_mlp_workspace_bytes(G, c_in, c_out, depth, N))
    L.check(lib.fgnn_debug_tc_mlp(L.PRECISIONS[prec], C.byref(p), L.ptr(xd), L.ptr(y), G, N,
                                  L.ptr(n_dev) if n_dev is not None else None, L.ptr(wsb), wsb.numel(),
                                  L.stream_ptr(DEV)), "fgnn_debug_tc_mlp")
    sd64 = {k: v.double() for k, v in sd.items()}
    tol = 2e-2 if prec == "bf16" else 3e-3
    for g in range(G):
        n = sizes[g] if sizes else N
        ref = O.mlp_block(x[g:g + 1, :, :n, :n].double(), sd64, "m", depth)[0]
        assert rel_fro(y[g, :, :n, :n].cpu(), ref) < tol
        assert float(y[g, :, n:, :].abs().sum()) == 0 and float(y[g, :, :, n:].abs().sum()) == 0


def feats(W):
    return torch.stack([O.adjacency_to_features(torch.from_numpy(w.astype(np.float32))) for w in W])


def build_model(z, precision, **extra):
    n, c, nb, depth, _ = [int(v) for v in z["meta"]]
    node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=nb,
                    in_features=c, out_features=c, depth_of_mlp=depth, **extra)
    model = pkg.models.Siamese_Node_Exp(2, node_emb)
    model.load_state_dict(state_dict_of(z))
    return model.to(DEV).set_precision(precision)


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("name", ["cfg1_er50_c32", "cfg3_reg40_c64"])
def test_tc_embedder_vs_reference_golden(name, prec):
    z = load_golden(name)
    model = build_model(z, prec)
    x1, x2 = feats(z["W1"]).to(DEV), feats(z["W2"]).to(DEV)
    with torch.no_grad():
        e1 = model.embed({"input": x1})
        scores = model({"input": x1}, {"input": x2})
    err = rel_fro(e1.cpu(), z["emb1"])
    print(f"{name} {prec}: embedding rel err {err:.3e}")
    assert err < EMB_TOL[prec]
    assert rel_fro(scores.cpu(), z["scores"]) < 2 * EMB_TOL[prec]


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
def test_tc_ragged_embedder_vs_per_graph_oracle(prec):
    gen = torch.Generator().manual_seed(17)
    sizes = [50, 23, 37, 64, 130]
    sd = O.xavier_state_dict(2, 32, 3, 3, gen, randomize_gn=True)
    node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=3,
                    in_features=32, out_features=32, depth_of_mlp=3, constant_n_vertices=False)
    model = pkg.models.Siamese_Node_Exp(2, node_emb)
    model.load_state_dict(sd)
    model = model.to(DEV).set_precision(prec)
    graphs = [O.synthetic_pair(s, 0.3, 0.1, gen)[0] for s in sizes]
    refs = O.node_embedding_ragged([g.double() for g in graphs], {k: v.double() for k, v in sd.items()})
    with torch.no_grad():
        e = model.embed({"input": mt.from_list(graphs, dims=(1, 2)).to(DEV)})
    assert isinstance(e, mt.MaskedTensor) and e.tensor.names == ('B', None, 'N')
    et = e.tensor.rename(None).cpu()
    for i, s in enumerate(sizes):
        assert rel_fro(et[i, :, :s], refs[i]) < EMB_TOL[prec]
        assert float(et[i, :, s:].abs().sum()) == 0
        # a graph embedded inside a ragged batch == the same graph embedded alone
        with torch.no_grad():
            solo = model.embed({"input": graphs[i][None].to(DEV)})
        # (statistics are accumulated per thread in fp32 over a batch-dependent tile partition, so this is
        # equality up to the 16-bit rounding noise floor, not bitwise -- see DESIGN.md)
        assert rel_fro(solo[0].cpu(), et[i, :, :s]) < EMB_TOL[prec]


def unpack_adj(bits, n):
    return np.unpackbits(bits, axis=-1)[..., :n]


# Benched shapes against outputs of the UNMODIFIED reference (tests/golden, oracle/make_golden.py round2).
# north_star: 16-bit mode within 2e-2 relative on node embeddings.  fp16 (what bench.py runs) meets it at both
# shapes; bf16 does not on random-init weights (DESIGN.md "Precision") and asserts 1.2x its measured error.
BENCHED_TOL = {("cfg3_reg500_c64", "fp16"): 2e-2, ("cfg2_er200_c32", "fp16"): 2e-2,
               ("cfg3_reg500_c64", "bf16"): 1.25e-1, ("cfg2_er200_c32", "bf16"): 2.5e-1}


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("name", ["cfg3_reg500_c64", "cfg2_er200_c32"])
def test_benched_shapes_vs_reference_golden(name, prec):
    z = load_golden(name)
    n = int(z["meta"][0])
    model = build_model(z, prec)
    x1, x2 = feats(unpack_adj(z["W1_bits"], n)).to(DEV), feats(unpack_adj(z["W2_bits"], n)).to(DEV)
    with torch.no_grad():
        e1 = model.embed({"input": x1})
        e2 = model.embed({"input": x2})
        scores = model({"input": x1}, {"input": x2})
        solo = model.embed({"input": x1[:1]})
        big = O.synthetic_pair(n + 20, 0.2, 0.1, torch.Generator().manual_seed(5))[0]
        # padding invariance is a property of the per-graph-n normalisation (constant_n_vertices=False); with the
        # default flag a padded batch normalises with Nmax (layers.py:76-77) and legitimately differs
        ragged = build_model(z, prec, constant_n_vertices=False).node_embedder.forward_fused(
            mt.from_list([feats(unpack_adj(z["W1_bits"], n))[0], big], dims=(1, 2)).to(DEV), prec)
    err1, err2 = rel_fro(e1.cpu(), z["emb1"]), rel_fro(e2.cpu(), z["emb2"])
    errs = rel_fro(scores.cpu(), z["scores"])
    print(f"PARITY {name} {prec}: emb1 {err1:.3e} emb2 {err2:.3e} scores {errs:.3e}")
    tol = BENCHED_TOL[(name, prec)]
    assert err1 < tol and err2 < tol
    assert errs < 2.5 * tol
    # batch independence and padding invariance hold to the statistics' summation-order noise (fp32 partial sums
    # over a batch-dependent tile partition), far below the 16-bit rounding error
    assert rel_fro(solo[0].cpu(), e1[0].cpu()) < tol / 4
    rg = ragged.tensor.rename(None)
    assert rel_fro(rg[0, :, :n].cpu(), e1[0].cpu()) < tol / 2
    assert float(rg[0, :, n:].abs().sum()) == 0


@pytest.mark.parametrize("prec", ["fp32", "fp16", "bf16"])
def test_trained_weights_predictions_match_reference(prec):
    """Per-row argmax matchings and both accuracies on a briefly trained model (real margins), north_star clause
    'per-row argmax matchings and alignment accuracy agreeing'."""
    from graph_neural_net_b200.toolbox.metrics import accuracy_max, accuracy_linear_assignment
    z = load_golden("trained_er50_c32")
    model = build_model(z, prec)
    x1, x2 = feats(z["W1"]).to(DEV), feats(z["W2"]).to(DEV)
    with torch.no_grad():
        scores = model({"input": x1}, {"input": x2})
    err = rel_fro(scores.cpu(), z["scores"])
    agree = float((scores.argmax(-1).cpu().numpy() == z["argmax"]).mean())
    acc = accuracy_max(scores)
    lap = accuracy_linear_assignment(scores)
    print(f"PARITY trained {prec}: scores rel err {err:.3e}, argmax agreement {agree:.4f}, acc {acc} vs {list(z['acc'])}, "
          f"lap {lap} vs {list(z['acc_lap'])}")
    total = int(z["acc"][1])
    if prec == "fp32":
        assert err < 2e-4 and agree >= 0.995
        assert abs(acc[0] - int(z["acc"][0])) <= 2 and abs(lap[0] - int(z["acc_lap"][0])) <= 2
    else:
        lim = {"fp16": (3e-2, 0.97, 0.03), "bf16": (3e-1, 0.80, 0.15)}[prec]
        assert err < lim[0] and agree >= lim[1]
        assert abs(acc[0] - int(z["acc"][0])) <= lim[2] * total
        assert abs(lap[0] - int(z["acc_lap"][0])) <= lim[2] * total
    assert acc[1] == total and lap[1] == total


@pytest.mark.parametrize("prec", ["fp32", "fp16"])
def test_ragged_constant_n_vertices_default(prec):
    """ADVICE r1: constant_n_vertices=True modules fed a MaskedTensor (the reference's default) normalise with the
    PADDED size (layers.py:76-77); fixture from the reference's masked embedder."""
    z = load_golden("ragged_cstn_c16")
    nmax, c, nb, depth, _ = [int(v) for v in z["meta"]]
    sizes = [int(v) for v in z["sizes"]]
    node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=nb,
                    in_features=c, out_features=c, depth_of_mlp=depth)          # flag left at its default (True)
    model = pkg.models.Siamese_Node_Exp(2, node_emb)
    model.load_state_dict(state_dict_of(z))
    model = model.to(DEV).set_precision(prec)          # fp16: the width-16 fixture runs zero-padded to 32 channels
    graphs = [O.adjacency_to_features(torch.from_numpy(z[f"W1/{i}"].astype(np.float32))) for i in range(len(sizes))]
    x = mt.from_list(graphs, dims=(1, 2)).to(DEV)
    with torch.no_grad():
        e = model.embed({"input": x}).tensor.rename(None).cpu()
    tol = 1e-4 if prec == "fp32" else EMB_TOL[prec]
    for i, n in enumerate(sizes):
        assert rel_fro(e[i, :, :n], z["masked_cstn_emb1"][i, :, :n]) < tol
        assert float(e[i, :, n:].abs().sum()) == 0


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
def test_tc_ragged_constant_n_vs_oracle(prec):
    """constant_n_vertices=True on a ragged batch through the fused 16-bit embedder: per-graph oracle with n = Nmax."""
    gen = torch.Generator().manual_seed(23)
    sizes = [70, 41, 96]
    nmax = max(sizes)
    sd = O.xavier_state_dict(2, 32, 3, 3, gen, randomize_gn=True)
    node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=3,
                    in_features=32, out_features=32, depth_of_mlp=3)
    model = pkg.models.Siamese_Node_Exp(2, node_emb)
    model.load_state_dict(sd)
    model = model.to(DEV).set_precision(prec)
    graphs = [O.synthetic_pair(s, 0.3, 0.1, gen)[0] for s in sizes]
    sd64 = {k: v.double() for k, v in sd.items()}
    with torch.no_grad():
        e = model.embed({"input": mt.from_list(graphs, dims=(1, 2)).to(DEV)}).tensor.rename(None).cpu()
    for i, s in enumerate(sizes):
        ref = O.node_embedding(graphs[i][None].double(), sd64, n=float(nmax))[0]
        other = O.node_embedding(graphs[i][None].double(), sd64)[0]
        err = rel_fro(e[i, :, :s], ref)
        print(f"PARITY ragged constant-n n={s} {prec}: {err:.3e} (vs per-graph-n oracle {rel_fro(e[i, :, :s], other):.3e})")
        assert err < EMB_TOL[prec]
        assert float(e[i, :, s:].abs().sum()) == 0


def test_bench_sized_launches_are_stable():
    """Regression for the input-ring phase aliasing (DESIGN.md 4.2): it needed BENCH-sized launches -- dozens of
    n=500 graphs per conv-chain launch, so that every CTA runs hundreds of tiles and the consumer can catch up with
    the TMA loads -- and showed as a GPU fault or a deadlock, never in the small parity cases.  52 graphs (two
    chunks) are embedded several times; every run must finish, agree with the first one to rounding (statistics
    are reduced with atomics) and graph 0 / graph 51 must agree with embedding them alone."""
    gen = torch.Generator().manual_seed(99)
    n, c, G = 500, 64, 52
    sd = O.xavier_state_dict(2, c, 4, 3, gen)
    node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=4,
                    in_features=c, out_features=c, depth_of_mlp=3)
    model = pkg.models.Siamese_Node_Exp(2, node_emb)
    model.load_state_dict(sd)
    model = model.to(DEV)
    base = (torch.rand((4, n, n), generator=gen) < 0.2).float()
    base = torch.triu(base, 1)
    base = base + base.transpose(1, 2)
    x = torch.stack([O.adjacency_to_features(base[i % 4][torch.randperm(n, generator=gen)][:, torch.randperm(n, generator=gen)])
                     for i in range(G)]).to(DEV)
    with torch.no_grad():
        first = model.node_embedder.forward_fused(x, "bf16")
        torch.cuda.synchronize()
        for _ in range(4):
            again = model.node_embedder.forward_fused(x, "bf16")
            torch.cuda.synchronize()
            assert torch.isfinite(again).all()
            assert rel_fro(again.cpu(), first.cpu()) < 1e-3
        for i in (0, G - 1):
            solo = model.node_embedder.forward_fused(x[i:i + 1], "bf16")
            assert rel_fro(solo[0].cpu(), first[i].cpu()) < 1e-1


def test_ragged_large_sizes_vs_oracle():
    """cfg4-like ragged batch (n from 50 to 1000, width 64, 4 blocks): the fp16 tensor-core embedder against the
    CPU oracle graph by graph (fp32 torch, a few seconds per graph); padding rows must be exactly zero (the fused
    pooling only ever touches rows < n)."""
    gen = torch.Generator().manual_seed(4242)
    sizes = [1000, 333, 50, 640, 128, 129]
    c = 64
    sd = O.xavier_state_dict(2, c, 4, 3, gen)
    node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=4,
                    in_features=c, out_features=c, depth_of_mlp=3, constant_n_vertices=False)
    model = pkg.models.Siamese_Node_Exp(2, node_emb)
    model.load_state_dict(sd)
    model = model.to(DEV)
    graphs = [O.synthetic_pair(s, 0.2, 0.1, gen)[0] for s in sizes]
    x = mt.from_list(graphs, dims=(1, 2)).to(DEV)
    with torch.no_grad():
        e = model.node_embedder.forward_fused(x, "fp16").tensor.rename(None).cpu()
        refs = O.node_embedding_ragged(graphs, sd)
    for i, s in enumerate(sizes):
        err = rel_fro(e[i, :, :s], refs[i])
        print(f"PARITY ragged n={s}: fp16 vs oracle rel err {err:.3e}")
        assert err < (2e-2 if s >= 200 else EMB_TOL["fp16"])
        assert float(e[i, :, s:].abs().sum()) == 0


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
def test_embedder_from_adjacency_equals_embedder_from_features(prec):
    """SURVEY 8(f) row 2: feeding the uint8 adjacency (input planes built on the device) gives the same embeddings
    as the reference's fp32 (W, diag(deg)) features -- the planes are identical, so only the atomics' order in the
    statistics can differ."""
    gen = torch.Generator().manual_seed(11)
    sizes = [150, 97, 64]
    N = max(sizes)
    sd = O.xavier_state_dict(2, 32, 3, 3, gen)
    node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=3,
                    in_features=32, out_features=32, depth_of_mlp=3, constant_n_vertices=False)
    model = pkg.models.Siamese_Node_Exp(2, node_emb)
    model.load_state_dict(sd)
    model = model.to(DEV)
    adj = torch.zeros((len(sizes), N, N), dtype=torch.uint8)
    graphs = []
    for g, n in enumerate(sizes):
        W = torch.triu(torch.rand((n, n), generator=gen) < 0.2, 1)
        W = W | W.T
        adj[g, :n, :n] = W.to(torch.uint8)
        graphs.append(O.adjacency_to_features(W.float()))
    n_dev = torch.tensor(sizes, dtype=torch.int32, device=DEV)
    with torch.no_grad():
        ref = model.node_embedder.forward_fused(mt.from_list(graphs, dims=(1, 2)).to(DEV), prec).tensor.rename(None)
        out = model.node_embedder.forward_fused_adjacency(adj.to(DEV), prec, n_dev)
    assert rel_fro(out.cpu(), ref.cpu()) < 1e-3
    for g, n in enumerate(sizes):
        assert float(out[g, :, n:].abs().sum()) == 0


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("shape", [(3, 64, 200, None), (4, 32, 50, None), (5, 64, 300, [300, 17, 129, 256, 257]), (2, 64, 1000, [1000, 513])])
def test_fused_head_matches_torch(prec, shape):
    """fgnn_head_fwd (tensor-core E1^T E2 + row softmax CE + row argmax, models/trainers.py:67, toolbox/losses.py:27-33,
    toolbox/metrics.py:125-134) against torch fp64 on random embeddings: the 16-bit (hi, lo) operand split keeps the
    scores at fp32 accuracy in BOTH precisions, so the bar is the fp32 one (1e-4 relative), not the 16-bit one."""
    from graph_neural_net_b200 import _ops
    G, Cc, N, sizes = shape
    gen = torch.Generator().manual_seed(11)
    e1 = torch.randn((G, Cc, N), generator=gen)
    e2 = (0.7 * e1 + 0.5 * torch.randn((G, Cc, N), generator=gen))
    n_dev = None
    if sizes is not None:
        n_dev = torch.tensor(sizes, dtype=torch.int32, device=DEV)
        for g, n in enumerate(sizes):
            e1[g, :, n:] = 0
            e2[g, :, n:] = 0
    ce, correct, scores = _ops.head_fused(e1.to(DEV), e2.to(DEV), n_dev, prec, want_scores=True)
    ce2, correct2, none = _ops.head_fused(e1.to(DEV), e2.to(DEV), n_dev, prec, want_scores=False)
    assert none is None and torch.equal(ce, ce2) and torch.equal(correct, correct2)      # deterministic, scores optional
    for g in range(G):
        n = N if sizes is None else sizes[g]
        ref = e1[g, :, :n].double().t() @ e2[g, :, :n].double()
        got = scores[g].cpu().double()
        assert float((got[:n, :n] - ref).norm() / ref.norm()) < 1e-5
        assert float(got[n:, :].abs().max() if n < N else 0.0) == 0.0 and float(got[:, n:].abs().max() if n < N else 0.0) == 0.0
        ref_ce = float(torch.nn.functional.cross_entropy(ref, torch.arange(n), reduction="sum"))
        assert abs(float(ce[g]) - ref_ce) < 1e-4 * max(1.0, abs(ref_ce)), (g, float(ce[g]), ref_ce)
        assert int(correct[g]) == int((ref.argmax(1) == torch.arange(n)).sum())


def test_loss_and_accuracy_matches_forward_plus_loss():
    """Siamese_Node_Exp.loss_and_accuracy (fused head, no (B,N,N) scores) == forward() + triplet_loss + accuracy_max."""
    from graph_neural_net_b200.toolbox.losses import triplet_loss
    from graph_neural_net_b200.toolbox.metrics import accuracy_max
    z = load_golden("cfg1_er50_c32")
    model = build_model(z, "fp16")
    x1, x2 = feats(z["W1"]).to(DEV), feats(z["W2"]).to(DEV)
    with torch.no_grad():
        scores = model({"input": x1}, {"input": x2})
        loss_a = float(triplet_loss()(scores))
        acc_a = accuracy_max(scores)
        loss_b, ok_b, rows_b = model.loss_and_accuracy({"input": x1}, {"input": x2})
    assert abs(loss_a - float(loss_b)) < 1e-5 * max(1.0, abs(loss_a))
    assert int(ok_b) == int(acc_a[0]) and int(rows_b) == int(acc_a[1])
    # the adjacency-fed variant (input construction on the device) agrees with the feature-fed one to rounding
    a1 = torch.from_numpy(np.asarray(z["W1"])).to(torch.uint8).to(DEV)
    a2 = torch.from_numpy(np.asarray(z["W2"])).to(torch.uint8).to(DEV)
    loss_c, ok_c, rows_c = model.loss_and_accuracy_from_adjacency(a1, a2)
    assert abs(float(loss_c) - loss_a) < 1e-3 * max(1.0, abs(loss_a)) and int(rows_c) == int(rows_b)


def test_full_size_permutation_equivariance_and_batch_independence():
    """Size-independent properties at the BENCHED shape (regular n=500, C=64, fp16), where the CPU oracle costs seconds per
    graph: (1) relabelling the vertices of the input permutes the node embeddings, e(P A P^T)[:, pi(i)] = e(A)[:, i] -- the tile
    partition, the hole columns and the ones rows / columns all move with the permutation, so this exercises every layout;
    (2) a graph embedded inside a batch equals the same graph embedded alone (GraphNorm statistics are per graph).  Both hold
    up to the 16-bit rounding noise of a different summation order (tolerance = 1.2x measured)."""
    from graph_neural_net_b200.loaders.data_generator import generate_pairs_on_device, adjacency_batch_to_tensor_representation
    gen = torch.Generator().manual_seed(5)
    n, c = 500, 64
    sd = O.xavier_state_dict(2, c, 4, 3, gen)
    node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=4,
                    in_features=c, out_features=c, depth_of_mlp=3)
    model = pkg.models.Siamese_Node_Exp(2, node_emb)
    model.load_state_dict(sd)
    model = model.to(DEV).set_precision("fp16")
    a1, a2 = generate_pairs_on_device("Regular", 3, n, 0.2, 0.1, seed=77)
    perm = torch.randperm(n, generator=gen).to(DEV)
    a1p = a1[:, perm][:, :, perm]                      # (P A P^T)[i, j] = A[perm[i], perm[j]]
    with torch.no_grad():
        e = model.embed({"input": adjacency_batch_to_tensor_representation(a1)})
        ep = model.embed({"input": adjacency_batch_to_tensor_representation(a1p)})
        solo = model.embed({"input": adjacency_batch_to_tensor_representation(a1[1:2])})
    err_perm = rel_fro(ep.cpu(), e[:, :, perm].cpu())
    err_solo = rel_fro(solo[0].cpu(), e[1].cpu())
    print(f"PARITY n=500 fp16: permutation equivariance {err_perm:.3e}, batch independence {err_solo:.3e}")
    assert err_perm < 5e-3 and err_solo < 5e-3          # measured 2.0e-3 .. 3.1e-3 (varies with the tile partition)


@pytest.mark.parametrize("widths", [(48, 40, 2), (24, 32, 3), (32, 64, 3), (64, 20, 2)])
def test_tc_embedder_other_widths_run_zero_padded(widths):
    """in_features / out_features other than a uniform 32 or 64 (the reference allows any: models/blocks_emb.py:29-36 maps
    in_features -> out_features in the last block) run on the tensor-core path zero-padded to 32 / 64 channels; padded channels
    are exactly zero and are sliced off.  fp16 embedder vs the fp64 oracle on the model's own random-init state."""
    cin, cout, depth = widths
    torch.manual_seed(cin * 100 + cout)
    node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=3,
                    in_features=cin, out_features=cout, depth_of_mlp=depth, constant_n_vertices=False)
    model = pkg.models.Siamese_Node_Exp(2, node_emb)
    with torch.no_grad():                                  # non-trivial affine parameters and biases
        for k, p in model.named_parameters():
            if k.endswith("bias"):
                p.normal_(0.0, 0.1)
            elif "gn.weight" in k:
                p.add_(0.2 * torch.randn_like(p))
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    model = model.to(DEV).set_precision("fp16")
    gen = torch.Generator().manual_seed(3)
    sizes = [70, 41]
    graphs = [O.synthetic_pair(n, 0.3, 0.1, gen)[0] for n in sizes]
    x = mt.from_list(graphs, dims=(1, 2)).to(DEV)
    with torch.no_grad():
        e = model.embed({"input": x}).tensor.rename(None).cpu()
    assert e.shape == (2, cout, max(sizes))
    sd64 = {k: v.double() for k, v in sd.items()}
    for i, n in enumerate(sizes):
        ref = O.node_embedding(graphs[i][None].double(), sd64)[0]
        err = rel_fro(e[i, :, :n], ref)
        print(f"PARITY widths in={cin} out={cout} depth={depth} n={n}: fp16 vs fp64 oracle {err:.3e}")
        assert err < 1e-2          # measured 2.9e-3 .. 7.4e-3
        assert float(e[i, :, n:].abs().sum()) == 0
    # the siamese model end to end at this width: fused head (width padded to a multiple of 16) vs forward + loss
    from graph_neural_net_b200.toolbox.losses import triplet_loss
    x2 = mt.from_list([O.synthetic_pair(n, 0.3, 0.1, gen)[1] for n in sizes], dims=(1, 2)).to(DEV)
    with torch.no_grad():
        loss_b, ok_b, rows_b = model.loss_and_accuracy({"input": x}, {"input": x2})
        loss_a = float(triplet_loss()(model({"input": x}, {"input": x2})))
    assert abs(loss_a - float(loss_b)) < 1e-4 * max(1.0, abs(loss_a)) and int(rows_b) == sum(sizes)


def test_bench_line_carries_the_contract_keys(tmp_path):
    """bench.py (our arm) on the smallest workload: ONE JSON line with the contract's keys -- roofline of the dominant kernel
    (measured live with CUDA events), clocks sampled during the timed region, e2e from pinned host buffers with its byte
    counts, the count of our kernel launches -- and, with --dump-outputs, the last timed step's outputs as .npy files."""
    import json
    import os
    import subprocess
    import sys as _sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([_sys.executable, os.path.join(root, "bench.py"), "--steps", "3", "--warmup", "3", "--no-secondary",
                          "--no-cpu-baseline", "--workload", "cfg1_er_n50_c32_b32_fwd", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "roofline", "clocks", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["value"] > 0 and d["gpu_launches"] > 0 and d["dtype"] == "f16"
    r = d["roofline"]
    assert r["bound"] in ("tensor", "hbm") and 0 < r["frac"] < 1.05 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 2 * 32 * 2 * 50 * 50 * 4 and e["d2h_bytes_per_step"] == 8
    assert "sm_mhz" in d["clocks"] and "reasons" in d["clocks"]
    dumped = {k: np.load(tmp_path / f"{k}.npy") for k in ("ce_sum", "correct", "emb1", "emb2")}
    assert sorted(os.listdir(tmp_path)) == sorted(f"{k}.npy" for k in dumped)
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in dumped.values())
    assert dumped["ce_sum"].shape == dumped["correct"].shape == (32,) and dumped["emb1"].shape == dumped["emb2"].shape == (32, 32, 50)
    # the per-pair loss and accuracy are those of the dumped embeddings (the head is deterministic)
    ce, correct, _ = _ops.head_fused(torch.from_numpy(dumped["emb1"]).to(DEV), torch.from_numpy(dumped["emb2"]).to(DEV), None, "fp16")
    assert rel_fro(ce.cpu(), dumped["ce_sum"]) < 1e-6 and np.array_equal(correct.cpu().numpy(), dumped["correct"])
