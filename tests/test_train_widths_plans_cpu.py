"""CPU tests of the 16-bit plans for embedders whose widths are not a uniform 32 or 64: the library runs them zero-padded
to C = 32 or 64, so their workspaces are those of the uniform model of width C, and widths above 64 are refused."""
import ctypes

import pytest

from graph_neural_net_b200 import _lib as L

# (in_features, out_features, depth) as the GPU tests train them, and a few more
CASES = [(48, 40, 2), (24, 32, 3), (32, 64, 3), (64, 20, 2), (16, 16, 3), (32, 16, 3), (1, 1, 2), (64, 33, 1)]


def embed_params(cin0, in_f, out_f, depth, nb=3):
    """Shapes of node_embedding(cin0, nb, in_f, out_f, depth): block i maps widths[i] -> widths[i + 1]
    (models/blocks_emb.py); the planners read no parameter data."""
    widths = [cin0] + [in_f] * (nb - 1) + [out_f]
    p = L.EmbedParams()
    p.num_blocks = nb
    for b in range(nb):
        ci, co = widths[b], widths[b + 1]
        for name, c_in in (("mlp1", ci), ("mlp2", ci), ("mlp3", ci + co)):
            m = getattr(p.block[b], name)
            m.c_in, m.c_out, m.depth, m.eps, m.constant_n = c_in, co, depth, 1e-5, 1
    return p


def twin_width(in_f, out_f):
    return 32 if max(in_f, out_f) <= 32 else 64


@pytest.fixture(autouse=True)
def plan_env(monkeypatch):
    for v in ("FGNN_TC_TRAIN_WS_GB", "FGNN_TC_WS_GB", "FGNN_TC_CHUNK"):
        monkeypatch.delenv(v, raising=False)


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
@pytest.mark.parametrize("in_f,out_f,depth", CASES)
def test_padded_widths_take_the_twin_workspace(in_f, out_f, depth, prec):
    lib = L.get_lib()
    C = twin_width(in_f, out_f)
    for G, N in ((1, 50), (16, 200), (128, 200), (3, 1024)):
        for query in (lib.fgnn_embed_workspace_bytes, lib.fgnn_embed_train_workspace_bytes):
            mine = query(ctypes.byref(embed_params(2, in_f, out_f, depth)), L.PRECISIONS[prec], G, N)
            twin = query(ctypes.byref(embed_params(2, C, C, depth)), L.PRECISIONS[prec], G, N)
            assert mine == twin > 0, (query.__name__, G, N, mine, twin)


@pytest.mark.parametrize("in_f,out_f", [(65, 65), (32, 65), (65, 16), (128, 128), (128, 32)])
def test_widths_above_64_are_refused(in_f, out_f):
    lib = L.get_lib()
    p = embed_params(2, in_f, out_f, 2)
    assert lib.fgnn_embed_workspace_bytes(ctypes.byref(p), L.PRECISIONS["fp16"], 4, 100) == 0
    assert "up to 64" in lib.fgnn_last_error().decode()
    assert lib.fgnn_embed_train_workspace_bytes(ctypes.byref(p), L.PRECISIONS["fp16"], 4, 100) == 0
    assert "up to 64" in lib.fgnn_last_error().decode()


def test_widths_that_do_not_chain_are_refused():
    lib = L.get_lib()
    p = embed_params(2, 24, 40, 2)
    p.block[2].mlp3.c_out = 24                       # the block's three MLPs must share their output width
    assert lib.fgnn_embed_train_workspace_bytes(ctypes.byref(p), L.PRECISIONS["fp16"], 4, 100) == 0
    assert "same c_out" in lib.fgnn_last_error().decode()
    p = embed_params(2, 24, 40, 2)
    p.block[2].mlp3.c_in = 24 + 24                   # mlp3 reads cat[mult (40), block input (24)]
    assert lib.fgnn_embed_workspace_bytes(ctypes.byref(p), L.PRECISIONS["fp16"], 4, 100) == 0
    assert "do not chain" in lib.fgnn_last_error().decode()
