"""Pin the cross-attention oracle (SURVEY §8f N4) to golden vectors made by the LIVE reference's
MultiheadAttention on its static_kv / incremental path (oracle/make_golden_xattn.py)."""
import os

import pytest
import torch

from oracle import cross_attention_oracle as X
from oracle.golden import load as load_golden


@pytest.fixture(scope="module")
def golden(golden_dir):
    return load_golden(os.path.join(golden_dir, "xattn.pt"))


def _close(a, b, tol=2e-5):
    assert a.shape == b.shape
    assert (a - b).abs().max().item() <= tol * max(1.0, b.abs().max().item())


def test_full_call_matches_golden(golden):
    for name, c in golden.items():
        a, w = X.cross_attention(c["params"], c["H"], c["full"]["query"], c["encoder_out"],
                                 c["encoder_padding_mask"], None, True, c["need_head_weights"])
        _close(a, c["full"]["attn"])
        _close(w, c["full"]["weights"])


def test_incremental_steps_match_golden(golden):
    """Replication x beam, same-size reorders (the reference leaves the cache untouched: :416) and a
    shrinking batch, step by step."""
    for name, c in golden.items():
        U, beam = len(c["lens"]), c["beam"]
        order0 = torch.arange(U).view(-1, 1).repeat(1, beam).view(-1)
        eo, em = X.reorder_encoder_out(c["encoder_out"], c["encoder_padding_mask"], order0)
        state = {}
        for st in c["steps"]:
            if st["new_order"] is not None:
                X.reorder_state(state, st["new_order"])
                eo, em = X.reorder_encoder_out(eo, em, st["new_order"])
            a, w = X.cross_attention(c["params"], c["H"], st["query"], eo, em, state, True,
                                     c["need_head_weights"])
            _close(a, st["attn"])
            _close(w, st["weights"])


def test_masked_keys_get_zero_weight(golden):
    c = golden["beam2_shrink"]
    w = c["full"]["weights"]  # [bsz, tgt, S]
    for u, n in enumerate(c["lens"]):
        assert (w[u, :, n:] == 0).all()
        assert torch.allclose(w[u].sum(-1), torch.ones(3), atol=1e-5)


def test_same_size_reorder_is_a_noop_in_the_reference(golden):
    """The quirk the device path must reproduce: a same-size new_order does NOT permute the cached
    K/V (multihead_attention.py:416), because hypotheses of one utterance share them."""
    c = golden["beam2_shrink"]
    state = {"prev_key": torch.arange(6.0).view(6, 1, 1, 1)}
    X.reorder_state(state, torch.tensor([5, 4, 3, 2, 1, 0]))
    assert state["prev_key"].flatten().tolist() == [0, 1, 2, 3, 4, 5]
    X.reorder_state(state, torch.tensor([5, 0]))
    assert state["prev_key"].flatten().tolist() == [5, 0]
