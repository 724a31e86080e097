"""CPU tests of the host-side planning for graphs above 1024 vertices: workspace sizes, pass cutting and the limits that
stay (nothing here touches a device)."""
import ctypes

import pytest

from graph_neural_net_b200 import _lib as L


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


def ws(params, G, N, train=False):
    lib = L.get_lib()
    f = lib.fgnn_embed_train_workspace_bytes if train else lib.fgnn_embed_workspace_bytes
    return f(ctypes.byref(params), L.PRECISIONS["fp16"], G, N)


@pytest.mark.parametrize("c,graph_gb,per_pass", [(32, 5.8, 2), (64, 11.6, 1)])
def test_embed_passes_at_4096(c, graph_gb, per_pass, monkeypatch):
    """One graph of N = 4096 takes graph_gb GB of planes; the batch is cut into equal passes within FGNN_TC_WS_GB
    (default 16 GiB), never less than one graph per pass, and the workspace is that of one pass."""
    p = embed_params(c)
    monkeypatch.delenv("FGNN_TC_WS_GB", raising=False)
    monkeypatch.delenv("FGNN_TC_CHUNK", raising=False)
    one = ws(p, 1, 4096)
    assert abs(one / 1e9 - graph_gb) < 0.1
    assert ws(p, 6, 4096) == ws(p, per_pass, 4096) and ws(p, 5, 4096) == ws(p, per_pass, 4096)
    assert ws(p, per_pass, 4096) < 16 * 2**30 + 2**26
    monkeypatch.setenv("FGNN_TC_WS_GB", "6" if c == 32 else "12")   # a graph nearly fills the budget: one per pass
    assert ws(p, 6, 4096) == one
    monkeypatch.setenv("FGNN_TC_WS_GB", "1")                         # less than one graph: still one per pass
    assert ws(p, 6, 4096) == one


def test_embed_and_training_limits():
    p = embed_params(32)
    lib = L.get_lib()
    assert ws(p, 1, 4096) > 0
    assert ws(p, 1, 4097) == 0 and "N <= 4096" in lib.fgnn_last_error().decode()
    assert ws(p, 1, 1024, train=True) > 0
    assert ws(p, 1, 1025, train=True) == 0 and "N <= 1024" in lib.fgnn_last_error().decode()


def test_regular_generator_workspace_holds_the_bitmaps_above_1264():
    lib = L.get_lib()
    edges = lambda G, N: G * (N * N // 2 + 16) * 4
    align = lambda b: (b + 255) // 256 * 256
    for N in (50, 500, 1024, 1264):                           # bitmaps in shared memory: edge lists only, as before
        assert lib.fgnn_generate_workspace_bytes(3, N, 1) == align(edges(3, N))
    for N in (1265, 2048, 4096):
        assert lib.fgnn_generate_workspace_bytes(3, N, 1) == align(edges(3, N) + 3 * N * ((N + 31) // 32) * 4)
    assert lib.fgnn_generate_workspace_bytes(3, 4096, 0) == 256
