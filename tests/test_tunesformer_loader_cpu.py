"""TunesFormerShaped.load_reference_state_dict: the reference TunesFormer's state dict (HF GPT-2 parameter names, Conv1D
weights stored [in, out]) loads into the same parameters as the direct load the model tests use.  The HF names come from
oracle/make_golden_tunesformer.py::to_hf, the mapping that script checks against the unmodified reference's load_state_dict."""
import pytest
import torch

from oracle.make_golden_tunesformer import SPEC, inputs, to_hf


def _reference_sd(psd, csd):
    sd = to_hf(psd, "patch_level_decoder.base.")
    sd["patch_level_decoder.patch_embedding.weight"] = psd["patch_embedding.weight"].clone()
    sd["patch_level_decoder.patch_embedding.bias"] = psd["patch_embedding.bias"].clone()
    sd.update(to_hf(csd, "char_level_decoder.base.transformer."))
    sd["char_level_decoder.base.lm_head.weight"] = csd["transformer.wte.weight"].clone()
    # the attention mask buffers HF GPT-2 keeps in its state dict
    for prefix, n in (("patch_level_decoder.base.", SPEC["patch_cfg"]["n_layer"]),
                      ("char_level_decoder.base.transformer.", SPEC["char_cfg"]["n_layer"])):
        for i in range(n):
            sd[f"{prefix}h.{i}.attn.bias"] = torch.ones(1, 1, 4, 4)
            sd[f"{prefix}h.{i}.attn.masked_bias"] = torch.tensor(-1e4)
    return sd


def _models():
    from ai_music_generation_b200 import GPTConfig, TunesFormerShaped
    pc, cc, psd, csd, _ = inputs(SPEC)
    direct = TunesFormerShaped(GPTConfig(**SPEC["patch_cfg"]), GPTConfig(**SPEC["char_cfg"]))
    direct.patch_level_decoder.load_state_dict({**psd, "lm_head.weight": psd["transformer.wte.weight"]})
    direct.char_level_decoder.load_state_dict({**csd, "lm_head.weight": csd["transformer.wte.weight"]})
    torch.manual_seed(123)   # different initial weights: everything must come from the checkpoint
    loaded = TunesFormerShaped(GPTConfig(**SPEC["patch_cfg"]), GPTConfig(**SPEC["char_cfg"]))
    return direct, loaded, _reference_sd(psd, csd)


def test_reference_state_dict_loads_the_same_parameters():
    direct, loaded, sd = _models()
    assert loaded.load_reference_state_dict(sd) is loaded
    want, got = dict(direct.named_parameters()), dict(loaded.named_parameters())
    assert want.keys() == got.keys()
    for name, w in want.items():
        assert torch.equal(got[name].detach(), w.detach()), name
    for dec in (loaded.patch_level_decoder, loaded.char_level_decoder):   # the tie survives the load
        assert dec.lm_head.weight is dec.transformer.wte.weight


@pytest.mark.parametrize("edit", ["missing", "extra", "shape", "conv_shape", "shared_weights"])
def test_reference_state_dict_refuses_a_mismatch(edit):
    _, loaded, sd = _models()
    if edit == "missing":
        key = "char_level_decoder.base.transformer.h.1.mlp.c_fc.bias"
        del sd[key]
    elif edit == "extra":
        key = "patch_level_decoder.base.h.0.attn.c_attn.lora"
        sd[key] = torch.zeros(3)
    elif edit == "shape":
        key = "patch_level_decoder.patch_embedding.bias"
        sd[key] = torch.zeros(sd[key].numel() + 1)
    elif edit == "conv_shape":   # an untransposed Conv1D weight
        key = "char_level_decoder.base.transformer.h.0.attn.c_attn.weight"
        sd[key] = sd[key].t().contiguous()
    else:                        # one stack serving both levels: the character level's blocks are absent
        key = "char_level_decoder.base.transformer.h.0.ln_1.weight"
        sd = {k: v for k, v in sd.items() if not k.startswith("char_level_decoder.base.transformer.h.")}
    with pytest.raises((KeyError, ValueError), match=key.replace(".", r"\.")):
        loaded.load_reference_state_dict(sd)
