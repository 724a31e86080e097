"""CPU tests of the deterministic mode (FGNN_DETERMINISTIC): flag handling of the C ABI, the workspaces it asks for,
the plan choice that follows them, and a SASS audit of which kernels may add with floating-point atomics (nothing here
touches a device)."""
import ctypes
import os
import re
import shutil
import subprocess

import pytest

from graph_neural_net_b200 import _lib as L
from tests.test_train_plans_cpu import KEEP_ALL, embed_params

DET = L.FGNN_DETERMINISTIC
GIB = 2**30


@pytest.fixture(autouse=True)
def plan_env(monkeypatch):
    for v in ("FGNN_TC_TRAIN_WS_GB", "FGNN_TC_WS_GB", "FGNN_TC_CHUNK"):
        monkeypatch.delenv(v, raising=False)
    return monkeypatch


def lib():
    return L.get_lib()


def train_ws(c, G, N, prec):
    return lib().fgnn_embed_train_workspace_bytes(ctypes.byref(embed_params(c)), prec, G, N)


def infer_ws(c, G, N, prec):
    return lib().fgnn_embed_workspace_bytes(ctypes.byref(embed_params(c)), prec, G, N)


@pytest.mark.parametrize("prec", ["fp16", "bf16"])
def test_default_sizes_unchanged_and_deterministic_sizes_larger(prec, plan_env):
    plan_env.setenv("FGNN_TC_TRAIN_WS_GB", "1000")
    p = L.PRECISIONS[prec]
    for (n, c, g), nbytes in KEEP_ALL.items():
        assert train_ws(c, g, n, p) == nbytes, (n, c, g)
        assert train_ws(c, g, n, p | DET) > nbytes, (n, c, g)
    for n, c, g in ((50, 32, 16), (500, 64, 64), (2048, 32, 1), (4096, 64, 1)):
        base = infer_ws(c, g, n, p)
        assert base > 0 and infer_ws(c, g, n, p | DET) > base, (n, c, g)
    # the fp32 forward has no cross-CTA sums: the bit is accepted and changes nothing
    assert infer_ws(32, 4, 50, L.FP32 | DET) == infer_ws(32, 4, 50, L.FP32) > 0
    for args in ((16, 2, 32, 3, 50), (64, 64, 64, 3, 200)):
        base = lib().fgnn_mlp_workspace_bytes(*args)
        assert lib().fgnn_mlp_workspace_bytes_ex(*args, 0) == base
        assert lib().fgnn_mlp_workspace_bytes_ex(*args, DET) > base


def test_plan_choice_follows_the_deterministic_size(plan_env):
    """A keep-all threshold between the default and the deterministic keep-all sizes: the default keeps everything,
    the deterministic mode cuts the batch into recompute passes (of FGNN_TC_CHUNK graphs: smaller than keep-all)."""
    c, g, n = 32, 16, 200
    p = L.PRECISIONS["fp16"]
    plan_env.setenv("FGNN_TC_TRAIN_WS_GB", "1000")
    base, det = train_ws(c, g, n, p), train_ws(c, g, n, p | DET)
    assert base == KEEP_ALL[(n, c, g)] < det
    plan_env.setenv("FGNN_TC_TRAIN_WS_GB", repr((base + det) / 2 / GIB))
    plan_env.setenv("FGNN_TC_CHUNK", "4")
    assert train_ws(c, g, n, p) == base
    assert train_ws(c, g, n, p | DET) < base


@pytest.mark.parametrize("bad", [0x200, 0x1000, 1 << 30, -1])
def test_unknown_bits_are_rejected(bad):
    ep = ctypes.byref(embed_params(32))
    for prec in (L.FP16, L.BF16, L.FP32):
        assert lib().fgnn_embed_workspace_bytes(ep, prec | bad, 4, 50) == 0
        assert lib().fgnn_embed_train_workspace_bytes(ep, prec | bad, 4, 50) == 0
    assert lib().fgnn_mlp_workspace_bytes_ex(4, 2, 32, 3, 50, bad) == 0
    assert lib().fgnn_mlp_workspace_bytes_ex(4, 2, 32, 3, 50, bad | DET) == 0
    # the entry points refuse the flags before they look at anything else
    grads = L.EmbedGrads()
    calls = [
        lambda f: lib().fgnn_embed_fwd(ep, f, None, None, 4, 50, None, None, 0, None),
        lambda f: lib().fgnn_embed_fwd_adjacency_u8(ep, f, None, None, 4, 50, None, None, 0, None),
        lambda f: lib().fgnn_embed_fwd_train(ep, f, None, None, 4, 50, None, None, 0, None),
        lambda f: lib().fgnn_embed_bwd(ep, ctypes.byref(grads), f, None, 9, 4, 50, None, None, 0, None),
    ]
    for call in calls:
        assert call(L.FP16 | bad) == 1                     # FGNN_ERR_INVALID
        assert b"flags" in lib().fgnn_last_error()
        assert call(L.FP16 | DET) == 1                     # accepted: the call fails further on (null pointers)
        assert b"flags" not in lib().fgnn_last_error()
    mp, mg = L.MlpParams(), L.MlpGrads()
    assert lib().fgnn_mlp_bwd_f32_ex(ctypes.byref(mp), ctypes.byref(mg), None, None, None, None, 4, 50, None, None, 0,
                                     None, bad) == 1
    assert b"flags" in lib().fgnn_last_error()


# ---- SASS audit ----------------------------------------------------------------------------------------------------
# The default-mode kernels that sum partials from several CTAs with floating-point atomics (DESIGN.md "Deterministic
# mode"), each instantiated with the AtomicSum tag, and their OrderedSum twins that must contain no such instruction.
ATOMIC_KERNELS = {"tc_mlp_kernel", "gn_bwd_stats_kernel", "gn_bwd_apply_kernel", "relu_mask_kernel", "tc_wgrad_kernel",
                  "wgrad_kernel"}
FP_ATOMIC_ADD = re.compile(r"\b(?:RED|REDG|ATOM|ATOMG)\.[A-Z0-9_.]*ADD\.(?:F16|BF16|F16x2|BF16x2|F32|F64)\b")
BASE = re.compile(r"\d+(" + "|".join(sorted(ATOMIC_KERNELS, key=len, reverse=True)) + r")I")


def sass_functions():
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    if not os.path.exists(L.LIB_PATH):
        pytest.skip("library not built")
    out = subprocess.run([cuobjdump, "-sass", L.LIB_PATH], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            funcs[cur] = False
        elif cur is not None and FP_ATOMIC_ADD.search(line):
            funcs[cur] = True
    assert funcs, "no kernels in the SASS dump"
    return funcs


def test_sass_floating_point_atomics_only_in_default_mode_kernels():
    funcs = sass_functions()
    with_atomics = {f for f, has in funcs.items() if has}
    atomic_tagged = {f for f in funcs if "9AtomicSum" in f}
    ordered_tagged = {f for f in funcs if "10OrderedSum" in f}
    assert with_atomics == atomic_tagged, (sorted(with_atomics - atomic_tagged), sorted(atomic_tagged - with_atomics))
    assert not (with_atomics & ordered_tagged)
    # exactly the kernels of the list, each with its deterministic twin
    bases = {BASE.search(f).group(1) for f in atomic_tagged}
    assert bases == ATOMIC_KERNELS, bases
    assert {f.replace("9AtomicSum", "10OrderedSum") for f in atomic_tagged} == ordered_tagged
