"""Head sizes 32, 64 and 128 (n_embd // n_head), host side: config validation before any device allocation, the C ABI
entry points of csrc/attn_hd.cu, the replay id of the decode kernel, and plan recording of the new launches under the
existing attention names."""
import re

import pytest

from ai_music_generation_b200 import GPT, GPTConfig, _C, ops


def _cfg(n_embd, n_head):
    return GPTConfig(block_size=64, vocab_size=95, n_layer=1, n_head=n_head, n_embd=n_embd, dropout=0.0, bias=False)


@pytest.mark.parametrize("n_embd,n_head", [(384, 4), (96, 1), (256, 16), (768, 3)])
def test_unsupported_head_size_raises_value_error(n_embd, n_head):
    with pytest.raises(ValueError, match="32, 64, 128"):
        GPT(_cfg(n_embd, n_head))


def test_n_embd_not_divisible_by_n_head_raises_value_error():
    with pytest.raises(ValueError, match="multiple of n_head"):
        GPT(_cfg(100, 3))


@pytest.mark.parametrize("n_embd,n_head,D", [(128, 4, 32), (256, 8, 32), (256, 2, 128), (512, 4, 128), (768, 6, 128),
                                              (128, 2, 64)])
def test_supported_head_sizes_construct(n_embd, n_head, D):
    m = GPT(_cfg(n_embd, n_head))
    assert m._head_size == D
    assert m.transformer.h[0].attn.c_attn.weight.shape == (3 * n_embd, n_embd)


def test_header_function_ids_agree_with_replay_table():
    with open(_C.HEADER_PATH) as f:
        text = f.read()
    ids = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define ABCGPT_FN_([A-Z0-9_]+) (\d+)", text)}
    assert ids["ATTN_DECODE_HD"] == 7
    names = {"GEMM": "abcgpt_gemm_bf16"}   # the one id that is not named after its function
    assert {names.get(k, "abcgpt_" + k.lower()): v for k, v in ids.items()} == _C.FN_IDS


def test_head_size_entry_points_declared_and_bound():
    declared = _C.declared_symbols()
    for name in ("abcgpt_attn_fwd_hd", "abcgpt_attn_bwd_hd", "abcgpt_attn_decode_hd"):
        assert name in declared and name in _C._SIGNATURES
    # dropout arguments stay last before the stream: ops.key_patches reads args[-3] / args[-2]
    for name in ("abcgpt_attn_fwd_hd", "abcgpt_attn_bwd_hd"):
        args = _C._SIGNATURES[name][1]
        assert args[-3] is _C.c_float and args[-2] is _C.c_uint32


def test_head_size_launches_record_under_attention_names(monkeypatch):
    """The _hd launches are recorded as "attn_fwd" / "attn_bwd", so a training plan's dropout keys are patched at replay."""
    calls = []

    class FakeLib:
        def __getattr__(self, name):
            def fn(*args):
                calls.append(name)
                return 0
            fn.__name__ = name
            return fn

    class T:
        def __init__(self):
            self.is_cuda, self.dtype = True, __import__("torch").bfloat16

        def data_ptr(self):
            return 4096

    monkeypatch.setattr(_C, "lib", lambda: FakeLib())
    monkeypatch.setattr(ops, "_stream", lambda: 0)
    ops.begin_record()
    ops.attn_fwd(T(), T(), T(), 2, 100, 4, drop_p=0.2, drop_key=11, head_size=32)
    ops.attn_bwd(T(), T(), T(), T(), T(), T(), 2, 100, 4, drop_p=0.2, drop_key=11, head_size=128)
    ops.attn_fwd(T(), T(), T(), 2, 100, 4, drop_p=0.2, drop_key=22, head_size=64)
    plan = ops.end_record()
    assert calls == ["abcgpt_attn_fwd_hd", "abcgpt_attn_bwd_hd", "abcgpt_attn_fwd"]
    assert [e[0] for e in plan] == ["attn_fwd", "attn_bwd", "attn_fwd"]
    assert plan[0][3][6] == 32 and plan[1][3][9] == 128
    patches = ops.key_patches(plan, [11, 22])
    assert patches == [(0, 0), (1, 0), (2, 1)]
