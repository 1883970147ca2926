"""Per-kernel parity on the GPU through the C ABI (ctypes -> libabcgpt.so), each kernel against a plain fp32
PyTorch statement of the same op.  The case definitions live in tools/gpu_probe.py (also used for timing)."""
import pytest

pytestmark = pytest.mark.gpu

from tools import gpu_probe  # noqa: E402

FAST_CASES = [
    "gemm_nt_small_bn128", "gemm_nt_small_bn256", "gemm_nn_small_bn128", "gemm_nn_small_bn256",
    "gemm_tn_small_bn128", "gemm_tn_small_bn256", "gemm_nt_k256_bn256", "gemm_nt_ragged", "gemm_nt_f32",
    "gemm2_nt_small", "gemm2_nt_k512", "gemm2_nn", "gemm2_tn", "gemm2_tn_red", "gemm2_ragged", "gemm2_gelu", "gemm2_resid",
    "gemm2_dgelu", "gemm2_half_nt", "gemm2_half_nn", "gemm2_half_gelu", "gemm2_half_dgelu", "gemm2_half_resid", "gemm_auto_cfg2_resid", "gemm_auto_cfg2_dgrad", "gemm_auto_cfg2_dgelu", "gemm_auto_cfg2_wgrad", "gemm2_gelu_tanh", "gemm2_dgelu_tanh", "gemm_gelu", "gemm_resid", "gemm_dgelu", "gemm_wgrad_red",
    "attn_spike", "attn_t32", "attn_t32_packed", "attn_t64_packed", "attn_t64", "attn_t128", "attn_t200", "attn_t256", "attn_t1024",
    "ln_384", "ln_768", "ln_768_bias", "ln_1000", "ln_resid_768", "ln_resid_1000_bias", "ce_95", "ce_50304", "colsum_768", "colsum_narrow_130", "adamw", "embed", "embed_bigv",
]


@pytest.mark.parametrize("name", FAST_CASES)
def test_kernel_case(name, cuda_device):
    res = gpu_probe.build_cases()[name]()
    assert res["ok"], res


def test_full_size_gemm_shapes(cuda_device):
    """BASELINE cfg3 shapes (M = 32*1024): bf16 rounding-level agreement with an fp32 matmul."""
    cases = gpu_probe.build_cases()
    for name in ("gemm_perf_c_attn", "gemm_perf_mlp_proj_resid", "gemm_perf_dgrad_proj_dgelu", "gemm_perf_wgrad_fc",
                 "gemm_perf_lm_head"):
        res = cases[name]()
        assert res["ok"], res


def test_missing_cuda_tensor_is_loud(cuda_device):
    import torch
    from ai_music_generation_b200 import _C, ops
    with pytest.raises(_C.AbcgptError):
        ops.gemm(torch.zeros(128, 64, dtype=torch.bfloat16), torch.zeros(128, 64, dtype=torch.bfloat16),
                 out=torch.zeros(128, 128, dtype=torch.bfloat16))


def test_pair_gemm_dynamic_tile_scheduler(cuda_device, tmp_path):
    """Opt-in ticket-based tile scheduler of the CTA-pair GEMM (ABCGPT_DYNAMIC_TILES=1, read once per process): the same
    parity cases in a child process, including split-K wgrad (work items = tiles x splits) and the full cfg3 shapes (5-21
    tiles per pair, several trips around the 16-slot ring)."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    names = ["gemm2_nt_small", "gemm2_nt_k512", "gemm2_nn", "gemm2_tn_red", "gemm2_ragged", "gemm2_gelu", "gemm2_resid",
             "gemm_perf_c_attn", "gemm_perf_c_fc_gelu", "gemm_perf_wgrad_fc", "gemm_perf_dgrad_fc"]
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "gpu_probe.py"), *names],
                       env=dict(os.environ, ABCGPT_DYNAMIC_TILES="1", ABCGPT_PROBE_OUT=str(tmp_path)), capture_output=True,
                       text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    import re
    m = re.search(r"PROBE SUMMARY: (\d+)/(\d+) ok", r.stdout)   # names select by prefix (gemm2_gelu also runs gemm2_gelu_tanh)
    assert m and m.group(1) == m.group(2) and int(m.group(2)) >= len(names) and "failed: []" in r.stdout, r.stdout[-2000:]
