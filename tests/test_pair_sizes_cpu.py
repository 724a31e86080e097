"""Host-side checks of graph pairs of unequal sizes: per-dim MaskedTensor sizes, the (N1, N2) head workspace query and
the loss's refusal of pairs whose graph 1 is larger than graph 2.  No GPU needed."""
import pytest
import torch

from graph_neural_net_b200 import _lib as L
from graph_neural_net_b200.maskedtensors import maskedtensor as mt
from graph_neural_net_b200.toolbox.losses import _as_batch, check_loss_sizes, triplet_loss


def scores_like(n1, n2):
    """Scores of pairs (n1[g], n2[g]) as a MaskedTensor whose rows and columns carry different masks."""
    return mt.from_list([torch.ones(a, b) for a, b in zip(n1, n2)], dims=(0, 1))


def test_per_dim_sizes():
    s = scores_like([3, 5, 2], [4, 6, 2])
    assert s.sizes_host("N") == [3, 5, 2]
    assert s.sizes_host("N_") == [4, 6, 2]
    assert s.sizes_i32(name="N_").dtype == torch.int32 and s.sizes_i32(name="N_").tolist() == [4, 6, 2]
    with pytest.raises(ValueError, match="same size"):
        s.sizes_host()
    with pytest.raises(KeyError):
        s.sizes_host("M")
    t, n1, n2, rows = _as_batch(s)
    assert t.shape == (3, 5, 6) and n1.tolist() == [3, 5, 2] and n2.tolist() == [4, 6, 2] and rows.tolist() == [3, 5, 2]


def test_per_dim_sizes_need_prefix_masks():
    s = scores_like([3, 5], [4, 6])
    s.mask_dict["N_"] = torch.tensor([[1., 0., 1., 1., 0., 0.], [1.] * 6]).refine_names("B", "N_")
    with pytest.raises(ValueError, match="prefix"):
        s.sizes_host("N_")


def test_equal_sizes_keep_the_shared_size():
    s = scores_like([3, 5], [3, 5])
    assert s.sizes_host() == [3, 5] == s.sizes_host("N") == s.sizes_host("N_")


@pytest.mark.parametrize("G", [1, 7, 64, 65535])
@pytest.mark.parametrize("N1", [1, 50, 128, 129, 1000, 4096])
def test_pair_workspace_depends_on_rows_only(G, N1):
    lib = L.get_lib()
    assert lib.fgnn_head_pair_workspace_bytes(G, N1) == lib.fgnn_head_workspace_bytes(G, N1)
    assert lib.fgnn_head_workspace_bytes(G, N1) == -(-G * -(-N1 // 128) * 8 // 256) * 256


def test_loss_refuses_more_rows_than_columns():
    with pytest.raises(ValueError, match=r"n1=5 > n2=3"):
        triplet_loss()(torch.zeros(2, 5, 3))
    with pytest.raises(ValueError, match=r"pair 1 has n1=6 > n2=4"):
        triplet_loss()(scores_like([3, 6], [4, 4]))
    check_loss_sizes([3, 4], [3, 9])


def test_loss_accepts_fewer_rows_than_columns_up_to_the_device():
    # the host checks pass; the call then fails on the missing CUDA tensor (there is no CPU fallback)
    with pytest.raises(L.FgnnError, match="CUDA"):
        triplet_loss()(torch.zeros(2, 3, 5))
