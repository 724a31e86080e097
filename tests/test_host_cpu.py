"""CPU tests: host logic of the reference-facing mirror and the C-ABI export surface."""
import copy
import ctypes
import os
import re

import numpy as np
import pytest
import torch
import yaml

import graph_neural_net_b200 as pkg
from graph_neural_net_b200 import _lib
from graph_neural_net_b200.maskedtensors import maskedtensor as mt
from tests.helpers import load_golden, state_dict_of

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def default_cfg():
    return yaml.safe_load(open(os.path.join(ROOT, "graph_neural_net_b200", "default_config.yaml")))


def test_shared_library_exports_every_declared_symbol():
    header = open(_lib.HEADER_PATH).read()
    declared = set(re.findall(r"\b(fgnn_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 20
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/fgnn_b200.h but not exported"
    assert set(_lib._SIGNATURES) == declared
    assert b"sm_100a" in pkg.get_lib().fgnn_version()


def test_config_keys_and_state_dict_layout():
    cfg = default_cfg()
    assert cfg["arch"]["original_features_num"] == 2
    for k in ("type", "block_init", "block_inside", "num_blocks", "in_features", "out_features",
              "depth_of_mlp", "num_heads"):
        assert k in cfg["arch"]["node_emb"]
    for k in ("lr", "scheduler_step", "scheduler_decay", "lr_stop", "batch_size", "epochs", "log_freq"):
        assert k in cfg["train"]
    model = pkg.models.get_siamese_model_exp(copy.deepcopy(cfg["arch"]), cfg["train"])
    sd = model.state_dict()
    assert len(sd) == 96 and sum(p.numel() for p in model.parameters()) == 40000
    ref = state_dict_of(load_golden("cfg1_er50_c32"))          # keys/shapes written by the reference
    assert set(sd) == set(ref)
    for k in sd:
        assert tuple(sd[k].shape) == tuple(ref[k].shape), k
    model.load_state_dict(ref)                                  # reference checkpoints load unchanged
    opt = model.configure_optimizers()
    assert isinstance(opt["optimizer"], torch.optim.Adam) and opt["lr_scheduler"]["monitor"] == "val_loss"


def test_network_graph_matches_reference_dag():
    cfg = default_cfg()
    model = pkg.models.get_siamese_model_exp(copy.deepcopy(cfg["arch"]), cfg["train"])
    keys = list(model.node_embedder.graph.keys())
    assert keys[:3] == ["input", "ne/in", "ne/bm/in"] and keys[-1] == "ne/suffix" and len(keys) == 28
    g = model.node_embedder.graph
    assert g["ne/bm/block2/mult"][1] == ["ne/bm/block2/mlp1", "ne/bm/block2/mlp2"]
    assert g["ne/bm/block2/cat"][1] == ["ne/bm/block2/mult", "ne/bm/block2/in"]
    assert g["ne/bm/block2/mlp3"][1] == ["ne/bm/block2/cat"]
    assert g["ne/bm/block2/in"][1] == ["ne/bm/block1/mlp3"]
    assert model.node_embedder._fused is not None and len(model.node_embedder._fused[2]) == 4


def test_unknown_registry_entries_raise_like_the_reference():
    cfg = default_cfg()
    for key in ("type", "block_inside", "block_init"):
        arch = copy.deepcopy(cfg["arch"])
        arch["node_emb"][key] = "nope"
        with pytest.raises(NotImplementedError):
            pkg.models.get_siamese_model_exp(arch, cfg["train"])
    with pytest.raises(ValueError):
        pkg.toolbox.losses.triplet_loss(loss_reduction="sum")


def test_from_list_matches_reference_padding_and_masks():
    z = load_golden("ragged_c16")
    sizes = [int(s) for s in z["sizes"]]
    from oracle import fgnn_oracle as O
    g1 = [O.adjacency_to_features(torch.from_numpy(z[f"W1/{i}"].astype(np.float32))) for i in range(len(sizes))]
    m = mt.from_list(g1, dims=(1, 2), base_name="N")
    assert m.tensor.names == ("B", None, "N", "N_")
    assert torch.equal(m.tensor.rename(None), torch.from_numpy(z["masked_input1"]))
    assert torch.equal(m.mask_dict["N"].rename(None), torch.from_numpy(z["mask_N"]))
    assert m.mask_dict["N_"].names == ("B", "N_")
    assert m.sizes_host() == sizes and len(m) == len(sizes)
    for i, g in enumerate(m):
        assert torch.equal(g, g1[i])
    # generic torch functions go through __torch_function__ and re-mask (API compatibility path)
    shifted = torch.add(m, 1.0)
    assert float(shifted.tensor.rename(None)[3, :, sizes[3]:, :].abs().max()) == 0
    mean = torch.mean(m)
    assert torch.allclose(mean.rename(None)[2], g1[2].mean(dim=(1, 2)))
    mx, _ = torch.max(m, 3)
    assert torch.equal(mx.tensor.rename(None)[1, :, :sizes[1]], g1[1].max(-1)[0])
    perm = m.permute(0, 1, 3, 2)
    assert perm.tensor.names == ("B", None, "N_", "N")
    bad = mt.MaskedTensor(m.tensor, {k: v.rename(None).flip(1).rename(*v.names) for k, v in m.mask_dict.items()}, adjust_mask=False)
    with pytest.raises(ValueError):
        bad.sizes_host()


def test_collate_functions():
    from graph_neural_net_b200.loaders.loaders import collate_fn_pair, collate_fn_pair_explore
    a = [(torch.ones(2, 3, 3), torch.zeros(2, 3, 3)), (torch.ones(2, 5, 5), torch.zeros(2, 5, 5))]
    m1, m2 = collate_fn_pair(a)
    assert m1.tensor.names == ("B", None, "N", "N_") and m2.tensor.names == ("B", None, "M", "M_")
    b = [(torch.ones(2, 4, 4), torch.zeros(2, 4, 4))] * 3
    d1, d2 = collate_fn_pair_explore(b)
    assert d1["input"].shape == (3, 2, 4, 4) and float(d2["input"].sum()) == 0


def test_install_as_reference_aliases():
    pkg.install_as_reference()
    import models.layers as ml          # noqa: E402  (alias of graph_neural_net_b200.models.layers)
    import maskedtensor as top_mt       # noqa: E402
    from toolbox.losses import triplet_loss  # noqa: E402,F401
    assert ml.MlpBlock_Real is pkg.models.layers.MlpBlock_Real and top_mt.from_list is mt.from_list


def test_device_side_input_construction_fails_loudly_off_gpu():
    """No CPU fallback: the adjacency entry points reject CPU tensors / unsupported precisions with FgnnError."""
    from graph_neural_net_b200._lib import FgnnError
    from graph_neural_net_b200.loaders import data_generator as dg
    adj = torch.zeros((2, 8, 8), dtype=torch.uint8)
    with pytest.raises(FgnnError):
        dg.adjacency_batch_to_tensor_representation(adj)
    cfg = default_cfg()
    model = pkg.models.get_siamese_model_exp(copy.deepcopy(cfg["arch"]), cfg["train"])
    with pytest.raises(FgnnError):
        model.node_embedder.forward_fused_adjacency(adj, "fp32")
    with pytest.raises(FgnnError):
        model.node_embedder.forward_fused_adjacency(adj, "bf16")
    # the host-side reference construction is unchanged
    W = torch.tensor([[0., 1., 1.], [1., 0., 0.], [1., 0., 0.]])
    B = dg.adjacency_matrix_to_tensor_representation(W)
    assert torch.equal(B[0], W) and torch.equal(B[1], torch.diag(torch.tensor([2., 1., 1.])))


def test_lightning_checkpoint_loads_through_get_siamese_model_test(tmp_path):
    """SURVEY 8(f) row 3: a Lightning-format checkpoint ({'state_dict': ...}, as written by the reference's Trainer) and a
    bare state dict both load through get_siamese_model_test (reference models/__init__.py:19-24), with the config
    found next to the run directory exactly as the reference looks it up."""
    import json
    from graph_neural_net_b200.models import get_siamese_model_test
    z = load_golden("tiny_er12_c8")
    n, c, nb, depth, _ = [int(v) for v in z["meta"]]
    sd = state_dict_of(z)
    node_emb = dict(type="node_embedding", block_init="block_emb", block_inside="block", num_blocks=nb,
                    in_features=c, out_features=c, depth_of_mlp=depth)
    # reference layout (models/__init__.py:19-22): <run>/config.json and <run>/<project>/<id>/checkpoints/<name>.ckpt
    run = tmp_path / "run0" / "proj" / "abc123" / "checkpoints"
    run.mkdir(parents=True)
    (tmp_path / "run0" / "config.json").write_text(json.dumps({"arch": {"original_features_num": 2, "node_emb": node_emb}}))
    for name, payload in (("lightning.ckpt", {"state_dict": sd, "epoch": 3, "pytorch-lightning_version": "1.9.0"}), ("bare.ckpt", sd)):
        torch.save(payload, run / name)
        model = get_siamese_model_test(str(run / name))
        got = model.state_dict()
        assert set(got) == set(sd)
        for k in sd:
            assert torch.equal(got[k], sd[k]), k
    cfg = {"arch": {"node_emb": node_emb}}
    model = get_siamese_model_test(str(run / "bare.ckpt"), config=cfg)
    assert torch.equal(model.state_dict()["node_embedder.ne_bm_block1_mlp1.convs.0.weight"],
                       sd["node_embedder.ne_bm_block1_mlp1.convs.0.weight"])


def test_bench_dump_outputs_samples_the_same_pairs_under_the_limit(tmp_path, monkeypatch):
    """bench.dump_outputs: float64 stays float64, the rest is stored as float32; above the size limit every per-pair array
    keeps the same seeded sample of pairs (identical from call to call), listed in pair_index.npy."""
    import bench
    gen = torch.Generator().manual_seed(1)
    arrays = {"ce_sum": torch.rand(40, generator=gen), "correct": torch.arange(40, dtype=torch.int32),
              "emb1": torch.rand((40, 8, 200), generator=gen), "loss": torch.tensor(0.5, dtype=torch.float64)}
    bench.dump_outputs(str(tmp_path / "all"), arrays)
    assert sorted(os.listdir(tmp_path / "all")) == ["ce_sum.npy", "correct.npy", "emb1.npy", "loss.npy"]
    assert np.array_equal(np.load(tmp_path / "all" / "emb1.npy"), arrays["emb1"].numpy())
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 200_000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b")) and "pair_index.npy" in names
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in names) <= 200_000
    a = {f[:-4]: np.load(tmp_path / "a" / f) for f in names}
    assert all(np.array_equal(v, np.load(tmp_path / "b" / f"{k}.npy")) for k, v in a.items())
    idx = a["pair_index"].astype(np.int64)
    assert 0 < len(idx) < 40 and np.all(np.diff(idx) > 0) and a["pair_index"].dtype == np.float64
    assert a["correct"].dtype == np.float32 and np.array_equal(a["correct"], idx)
    assert np.array_equal(a["emb1"], arrays["emb1"].numpy()[idx]) and np.array_equal(a["ce_sum"], arrays["ce_sum"].numpy()[idx])
    assert a["loss"].dtype == np.float64 and float(a["loss"]) == 0.5


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours) on the smallest workload: ONE JSON line with the
    contract's keys, `impl: reference`, an e2e object without copies, and a cpu_baseline that says which implementation was
    timed (the unmodified reference through oracle/refshim.py when its tree is present, else the oracle port)."""
    import json
    import subprocess
    import sys as _sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([_sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--workload", "cfg1_er_n50_c32_b32_fwd"], capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "pairs/s" and d["value"] > 0 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
