"""CPU tests of how 16-bit training cuts a batch into passes (one pass, or several the backward re-runs): which passes a
shape gets, the workspace they ask for, and the limits that stay (nothing here touches a device)."""
import ctypes
import os

import pytest

from graph_neural_net_b200 import _lib as L

GIB = 2**30
# one-pass workspaces (fp16 and bf16, 4 blocks of depth 3), byte for byte what they were before passes existed:
# (N, C, G) -> bytes
KEEP_ALL = {
    (200, 32, 1): 171_729_920,          # cfg2 golden: one pair of n = 200
    (200, 32, 16): 2_738_777_088,
    (200, 32, 128): 21_906_066_432,     # cfg2 as benched: 128 pairs
    (500, 64, 64): 107_271_556_096,     # cfg3, the benched architecture: 64 pairs
    (984, 32, 1): 3_305_198_592,        # cfg4's largest graph
    (1024, 64, 1): 8_649_697_280,
}


def embed_params(c):
    """Shapes of the default 4-block, depth-3 embedder (the workspace planners read no parameter data)."""
    p = L.EmbedParams()
    p.num_blocks = 4
    for b in range(4):
        cin = 2 if b == 0 else c
        for name, ci in (("mlp1", cin), ("mlp2", cin), ("mlp3", cin + c)):
            m = getattr(p.block[b], name)
            m.c_in, m.c_out, m.depth, m.eps, m.constant_n = ci, c, 3, 1e-5, 1
    return p


@pytest.fixture(autouse=True)
def plan_env(monkeypatch):
    for v in ("FGNN_TC_TRAIN_WS_GB", "FGNN_TC_WS_GB", "FGNN_TC_CHUNK"):
        monkeypatch.delenv(v, raising=False)
    return monkeypatch


def ws(c, G, N, prec="fp16"):
    return L.get_lib().fgnn_embed_train_workspace_bytes(ctypes.byref(embed_params(c)), L.PRECISIONS[prec], G, N)


def keep_all(monkeypatch, c, G, N):
    t = os.environ.get("FGNN_TC_TRAIN_WS_GB")
    monkeypatch.setenv("FGNN_TC_TRAIN_WS_GB", "100000")
    try:
        return ws(c, G, N)
    finally:
        if t is None:
            monkeypatch.delenv("FGNN_TC_TRAIN_WS_GB")
        else:
            monkeypatch.setenv("FGNN_TC_TRAIN_WS_GB", t)


def input_planes(G, N, cin=2):
    """Bytes of G graphs' 16-bit layout-C input planes (the workspace keeps them for the whole batch)."""
    bn = 64 if N <= 63 else (128 if N <= 127 else 256)
    npc = bn * -(-N // (bn - 1))
    return -(-G * cin * N * npc * 2 // 1024) * 1024


def pass_bytes(monkeypatch, c, G, N):
    """The part of the workspace that holds one pass of G graphs: their one-pass carve without their input planes."""
    return keep_all(monkeypatch, c, G, N) - input_planes(G, N)


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
def test_keep_all_is_unchanged_below_the_threshold(prec, plan_env):
    plan_env.setenv("FGNN_TC_TRAIN_WS_GB", "1000")
    for (n, c, g), nbytes in KEEP_ALL.items():
        assert ws(c, g, n, prec) == nbytes, (n, c, g)
    # T unset: half the device's memory, or unlimited without a device.  Far below half of any device: unchanged.
    plan_env.delenv("FGNN_TC_TRAIN_WS_GB")
    for g in (1, 16):
        assert ws(32, g, 200, prec) == KEEP_ALL[(200, 32, g)]


def test_recompute_workspace_is_one_pass_plus_the_input_planes(plan_env):
    plan_env.setenv("FGNN_TC_TRAIN_WS_GB", "1")
    got = ws(64, 64, 500)
    assert 0 < got < 20e9 < KEEP_ALL[(500, 64, 64)]
    # the largest pass within FGNN_TC_WS_GB (default 16 GiB), cut into equal passes
    cmax = max(k for k in range(1, 65) if pass_bytes(plan_env, 64, k, 500) <= 16 * GIB)
    passes = -(-64 // cmax)
    chunk = -(-64 // passes)
    assert 1 < chunk < 64
    assert got == pass_bytes(plan_env, 64, chunk, 500) + input_planes(64, 500)
    assert got <= keep_all(plan_env, 64, chunk, 500) + input_planes(64, 500)


def test_pass_is_never_less_than_one_graph(plan_env):
    plan_env.setenv("FGNN_TC_TRAIN_WS_GB", "0")
    plan_env.setenv("FGNN_TC_WS_GB", "1")          # one graph of N = 1024, C = 64 alone takes 8.65 GB
    one = pass_bytes(plan_env, 64, 1, 1024)
    assert one > GIB
    for g in (1, 3, 8):
        assert ws(64, g, 1024) == one + input_planes(g, 1024)
    assert ws(64, 1, 1024) == KEEP_ALL[(1024, 64, 1)]    # one graph: one pass, whatever T


def test_passes_are_equal(plan_env):
    plan_env.setenv("FGNN_TC_TRAIN_WS_GB", "0")
    plan_env.setenv("FGNN_TC_WS_GB", "8")
    cmax = max(k for k in range(1, 65) if pass_bytes(plan_env, 64, k, 500) <= 8 * GIB)
    assert cmax >= 2
    one_graph = input_planes(1, 500)
    for k in (2, 3, 5):
        full, short = ws(64, k * cmax, 500), ws(64, k * cmax - 1, 500)
        assert full - short == one_graph, k          # same passes of cmax graphs, one graph less of input planes
    for g in range(1, 4 * cmax + 2):                 # G graphs in ceil(G / cmax) passes of equal size
        chunk = -(-g // -(-g // cmax))
        assert ws(64, g, 500) == pass_bytes(plan_env, 64, chunk, 500) + input_planes(g, 500), g


def test_chunk_override_sets_the_pass(plan_env):
    plan_env.setenv("FGNN_TC_TRAIN_WS_GB", "0")
    plan_env.setenv("FGNN_TC_CHUNK", "3")
    assert ws(32, 9, 200) == pass_bytes(plan_env, 32, 3, 200) + input_planes(9, 200)
    assert ws(32, 7, 200) == pass_bytes(plan_env, 32, 3, 200) + input_planes(7, 200)   # passes of 3, 3, 1
    assert ws(32, 8, 200) == pass_bytes(plan_env, 32, 3, 200) + input_planes(8, 200)   # 3, 3, 2


@pytest.mark.parametrize("t", [None, "0"])
def test_training_limit_holds_under_both_plans(t, plan_env):
    if t is not None:
        plan_env.setenv("FGNN_TC_TRAIN_WS_GB", t)
    assert ws(32, 1, 1024) > 0
    assert ws(32, 1, 1025) == 0 and "N <= 1024" in L.get_lib().fgnn_last_error().decode()
    assert ws(64, 4, 1025) == 0 and "N <= 1024" in L.get_lib().fgnn_last_error().decode()
