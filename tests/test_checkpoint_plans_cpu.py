"""CPU tests of the checkpoint plan of 16-bit training (FGNN_CHECKPOINT_BLOCKS): flag handling of the C ABI, the
workspace the plan asks for, how it cuts passes, and its limits (nothing here touches a device)."""
import ctypes

import pytest

from graph_neural_net_b200 import _lib as L
from tests.test_train_plans_cpu import KEEP_ALL, embed_params, input_planes

CKPT = L.FGNN_CHECKPOINT_BLOCKS
DET = L.FGNN_DETERMINISTIC
FP16 = L.PRECISIONS["fp16"]
GIB = 2**30


@pytest.fixture(autouse=True)
def plan_env(monkeypatch):
    for v in ("FGNN_TC_TRAIN_WS_GB", "FGNN_TC_WS_GB", "FGNN_TC_CHUNK"):
        monkeypatch.delenv(v, raising=False)
    return monkeypatch


def lib():
    return L.get_lib()


def ws(c, G, N, prec=FP16 | CKPT, params=None):
    p = params if params is not None else embed_params(c)
    return lib().fgnn_embed_train_workspace_bytes(ctypes.byref(p), prec, G, N)


def last_error():
    return lib().fgnn_last_error().decode()


def batch_part(N, C, nb=4):
    """Bytes one graph adds to the batch-wide part of the checkpoint carve: its 16-bit input planes, every block's
    pre-norm output, every MLP's GraphNorm coefficients (2 floats) and statistics (4 floats) per channel and the pooling
    arg-max.  Exact where every region is a multiple of the arena's alignment, as at the shapes used here."""
    psc = input_planes(1, N, cin=1) // 2
    return input_planes(1, N) + nb * C * psc * 2 + nb * 3 * C * 6 * 4 + C * N * 4


def test_flag_is_accepted_by_the_training_entry_points_only():
    ep = ctypes.byref(embed_params(32))
    grads = L.EmbedGrads()
    for extra in (0, DET):
        for prec in (L.FP16, L.BF16):
            assert ws(32, 4, 50, prec | CKPT | extra) > 0
        for call in (lambda f: lib().fgnn_embed_fwd_train(ep, f, None, None, 4, 50, None, None, 0, None),
                     lambda f: lib().fgnn_embed_bwd(ep, ctypes.byref(grads), f, None, 9, 4, 50, None, None, 0, None)):
            assert call(L.FP16 | CKPT | extra) == 1         # accepted: the call fails further on (null pointers)
            assert "flags" not in last_error()
        # the inference entry points and the fp32 MLP backward's flags reject it
        for prec in (L.FP16, L.BF16, L.FP32):
            assert lib().fgnn_embed_workspace_bytes(ep, prec | CKPT | extra, 4, 50) == 0
        for call in (lambda f: lib().fgnn_embed_fwd(ep, f, None, None, 4, 50, None, None, 0, None),
                     lambda f: lib().fgnn_embed_fwd_adjacency_u8(ep, f, None, None, 4, 50, None, None, 0, None)):
            assert call(L.FP16 | CKPT | extra) == 1         # FGNN_ERR_INVALID
            assert "flags" in last_error()
        assert lib().fgnn_mlp_workspace_bytes_ex(4, 2, 32, 3, 50, CKPT | extra) == 0
    # fp32 has no 16-bit training workspace, with or without the flag
    assert ws(32, 4, 50, L.FP32 | CKPT) == 0


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
def test_smaller_than_keep_all_and_default_sizes_unchanged(prec, plan_env):
    plan_env.setenv("FGNN_TC_TRAIN_WS_GB", "1000")
    p = L.PRECISIONS[prec]
    for (n, c, g), nbytes in KEEP_ALL.items():
        assert ws(c, g, n, p) == nbytes, (n, c, g)
        got = ws(c, g, n, p | CKPT)
        assert 0 < got < nbytes, (n, c, g, got)
    # one graph: the checkpoint carve keeps about 24 plane sets of the 51 keep-all keeps
    assert ws(64, 1, 1024, p | CKPT) < 0.5 * KEEP_ALL[(1024, 64, 1)]


def test_train_ws_gb_plays_no_part(plan_env):
    ref = {(n, c, g): ws(c, g, n) for (n, c, g) in KEEP_ALL}
    for t in ("0", "1", "100000"):
        plan_env.setenv("FGNN_TC_TRAIN_WS_GB", t)
        for (n, c, g), nbytes in ref.items():
            assert ws(c, g, n) == nbytes, (t, n, c, g)


@pytest.mark.parametrize("n,c,gb", [(200, 32, 1), (500, 64, 8)])
def test_passes_are_equal_and_add_one_graph_of_batch_part(n, c, gb, plan_env):
    plan_env.setenv("FGNN_TC_WS_GB", str(gb))
    one = batch_part(n, c)

    def pass_part(k):      # a batch of k graphs in one pass of k
        plan_env.setenv("FGNN_TC_CHUNK", str(k))
        r = ws(c, k, n) - k * one
        plan_env.delenv("FGNN_TC_CHUNK")
        return r

    cmax = max(k for k in range(1, 65) if pass_part(k) <= gb * GIB)
    assert 2 <= cmax < 64
    for k in (2, 3, 5):
        full, short = ws(c, k * cmax, n), ws(c, k * cmax - 1, n)
        assert full - short == one, k                # the same k passes of cmax graphs, one graph less of batch part
    for g in range(1, 3 * cmax + 2):                 # G graphs in ceil(G / cmax) passes of equal size
        chunk = -(-g // -(-g // cmax))
        assert ws(c, g, n) == pass_part(chunk) + g * one, g


def test_chunk_override_sets_the_pass(plan_env):
    one = batch_part(200, 32)
    plan_env.setenv("FGNN_TC_CHUNK", "3")
    three = ws(32, 3, 200) - 3 * one
    assert ws(32, 9, 200) == three + 9 * one
    assert ws(32, 7, 200) == three + 7 * one        # passes of 3, 3, 1
    assert ws(32, 8, 200) == three + 8 * one        # 3, 3, 2
    plan_env.setenv("FGNN_TC_CHUNK", "1")
    assert ws(32, 9, 200) == ws(32, 1, 200) + 8 * one < three + 9 * one
    plan_env.setenv("FGNN_TC_CHUNK", "100")          # more than the batch: one pass
    assert ws(32, 9, 200) > three + 9 * one


def test_deterministic_workspace_is_larger():
    for (n, c, g) in KEEP_ALL:
        base = ws(c, g, n)
        assert ws(c, g, n, FP16 | CKPT | DET) > base > 0, (n, c, g)


def test_limits():
    got = ws(64, 1, 4096)
    assert 0 < got < 60e9, got                      # the benched width at the largest padded size
    assert ws(32, 1, 2048) > 0 and ws(32, 1, 4095) > 0
    for c, g in ((32, 1), (64, 2)):
        assert ws(c, g, 4097) == 0 and "N <= 4096" in last_error()
    # the other limits stay
    p = embed_params(32)
    p.block[2].mlp3.depth = 2
    assert ws(32, 1, 200, params=p) == 0 and "same depth" in last_error()
    p = embed_params(32)
    for name in ("mlp1", "mlp2", "mlp3"):
        getattr(p.block[3], name).c_out = 65
    p.block[3].mlp3.c_in = 65 + 32
    assert ws(32, 1, 200, params=p) == 0
    p = embed_params(32)
    for name, ci in (("mlp1", 65), ("mlp2", 65), ("mlp3", 65 + 32)):
        getattr(p.block[0], name).c_in = ci
    assert ws(32, 1, 200, params=p) == 0
    # without the flag, 16-bit training still stops at 1024 and says how to go further
    assert ws(32, 1, 1024, FP16) > 0
    assert ws(32, 1, 1025, FP16) == 0
    msg = last_error()
    assert "N <= 1024" in msg and "FGNN_CHECKPOINT_BLOCKS" in msg
