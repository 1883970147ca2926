"""Host-side pieces of packed TunesFormer training (no GPU): the pack_tunes layout, the row tables of the character level,
the per-tune loss weights restated in numpy, and the input validation that runs before any launch."""
import numpy as np
import pytest
import torch

from ai_music_generation_b200 import GPTConfig, TunesFormerShaped, pack_tunes
from ai_music_generation_b200.tunesformer import PATCH_SIZE, packed_decode_rows


def _tiny(dropout_p=0.0, dropout_c=0.0, block=16):
    pc = GPTConfig(block_size=block, vocab_size=128, n_layer=1, n_head=2, n_embd=128, dropout=dropout_p, bias=True,
                   activation="gelu_tanh")
    cc = GPTConfig(block_size=32, vocab_size=128, n_layer=1, n_head=2, n_embd=128, dropout=dropout_c, bias=True,
                   activation="gelu_tanh")
    return TunesFormerShaped(pc, cc)


def test_pack_tunes_layout():
    g = torch.Generator().manual_seed(0)
    tunes = [torch.randint(0, 128, (n, PATCH_SIZE), generator=g) for n in (2, 5, 3)]
    patches, counts = pack_tunes([tunes[0], tunes[1].tolist(), tunes[2]])
    assert counts == [2, 5, 3]
    assert patches.dtype == torch.int64 and patches.shape == (10, PATCH_SIZE)
    assert torch.equal(patches, torch.cat(tunes))
    with pytest.raises(ValueError):
        pack_tunes([])


def test_packed_decode_rows_restated():
    counts = [2, 5, 12, 16, 3]
    src, tune = packed_decode_rows(counts)
    cu = np.concatenate([[0], np.cumsum(counts)])
    want_src, want_tune = [], []
    for i, c in enumerate(counts):
        for j in range(c - 1):          # patch j of tune i conditions patch j + 1 of the same tune
            want_src.append(cu[i] + j)
            want_tune.append(i)
    assert src.tolist() == want_src and tune.tolist() == want_tune
    assert src.dtype == np.int64 and tune.dtype == np.int32
    assert not set((cu[1:] - 1).tolist()) & set(src.tolist())   # no tune's last patch conditions anything


def _weights(targets, row_group, n_groups, V=128):
    """numpy restatement of abcgpt_ce_group_weights."""
    valid = (targets >= 0) & (targets < V)
    cnt = np.bincount(row_group[valid], minlength=n_groups)
    return np.where(valid, 1.0 / (n_groups * np.maximum(cnt[row_group], 1)), 0.0)


def test_group_weights_give_mean_of_tune_means():
    rng = np.random.default_rng(0)
    counts = [2, 5, 12]
    _, tune = packed_decode_rows(counts)
    row_group = np.repeat(tune, PATCH_SIZE)
    targets = rng.integers(-1, 128, size=row_group.size)
    row_loss = rng.random(row_group.size)
    w = _weights(targets, row_group, len(counts))
    means = [row_loss[(row_group == i) & (targets >= 0)].mean() for i in range(len(counts))]
    assert np.isclose((w * row_loss).sum(), np.mean(means))
    assert np.all(w[targets < 0] == 0.0)


@pytest.mark.parametrize("counts, rows, msg", [
    ([1, 5], 6, "at least 2 patches"),
    ([3, 17], 20, "block_size"),
    ([3, 5], 9, "sum to"),
    ([], 0, "empty"),
])
def test_packed_validation_errors(counts, rows, msg):
    model = _tiny()
    with pytest.raises(ValueError, match=msg):
        model(torch.zeros(rows, PATCH_SIZE, dtype=torch.int64), patch_counts=counts)


@pytest.mark.parametrize("which", ["patch", "char"])
def test_packed_refuses_dropout(which):
    model = _tiny(dropout_p=0.1 if which == "patch" else 0.0, dropout_c=0.1 if which == "char" else 0.0)
    with pytest.raises(ValueError, match="dropout"):
        model(torch.zeros(5, PATCH_SIZE, dtype=torch.int64), patch_counts=[2, 3])


def test_packed_rejects_dense_shape():
    with pytest.raises(ValueError, match="packed patches"):
        _tiny()(torch.zeros(1, 5, PATCH_SIZE, dtype=torch.int64), patch_counts=[2, 3])
