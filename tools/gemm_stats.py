"""Where does the tcgen05 GEMM wait?  Per-role mbarrier wait cycles (debug counters) for the cfg3 shapes."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ai_music_generation_b200 import _C, ops  # noqa: E402
_C.use_debug_lib()  # instrumentation entry points live in libabcgpt_debug.so (include/abcgpt_debug.h)

dev = "cuda"
M, C = 32768, 768
stats = torch.zeros(8, device=dev, dtype=torch.int64)
shapes = [("c_attn fwd", M, 3 * C, C, False, False, ops.EPI_BF16), ("c_fc gelu", M, 4 * C, C, False, False, ops.EPI_GELU),
          ("attn c_proj resid", M, C, C, False, False, ops.EPI_RESID), ("mlp c_proj resid", M, C, 4 * C, False, False, ops.EPI_RESID),
          ("dgrad fc", M, C, 4 * C, False, True, ops.EPI_BF16), ("dgrad proj dgelu", M, 4 * C, C, False, True, ops.EPI_DGELU),
          ("wgrad fc", 4 * C, C, M, True, True, ops.EPI_F32_RED), ("wgrad attn", 3 * C, C, M, True, True, ops.EPI_F32_RED)]
for name, m, n, k, amn, bmn, epi in shapes:
    for bn in (512,):
        A = torch.randn((k, m) if amn else (m, k), device=dev).bfloat16()
        B = torch.randn((k, n) if bmn else (n, k), device=dev).bfloat16()
        odt = torch.float32 if epi in (ops.EPI_RESID, ops.EPI_F32_RED) else torch.bfloat16
        out = torch.zeros(m, n, device=dev, dtype=odt)
        out2 = torch.zeros(m, n, device=dev, dtype=torch.bfloat16) if epi == ops.EPI_GELU else None
        aux = torch.randn(m, n, device=dev, dtype=torch.float32 if epi == ops.EPI_RESID else torch.bfloat16) if epi in (ops.EPI_RESID, ops.EPI_DGELU) else None
        if aux is not None and epi == ops.EPI_DGELU:
            aux = aux.bfloat16()
        run = lambda: ops.gemm(A, B, a_mn=amn, b_mn=bmn, epilogue=epi, out=out, out2=out2, aux=aux, tile_n=bn)
        for _ in range(3):
            run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            run()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 10
        stats.zero_()
        _C.lib().abcgpt_debug_gemm_stats(stats.data_ptr())
        run()
        torch.cuda.synchronize()
        _C.lib().abcgpt_debug_gemm_stats(0)
        s = stats.tolist()
        tot = max(s[5], 1)
        # pair kernels: only the leader CTA of a pair issues MMAs, so its wait fractions are relative to half of the CTA time
        print(f"{name:20s} bn={bn} {ms*1e3:7.1f} us {2.0*m*n*k/ms/1e9:7.1f} TF/s | of CTA time: producer-waits-empty {s[0]/tot:5.2f}  "
              f"mma-waits-full {2*s[1]/tot:5.2f}  mma-waits-tmem {2*s[2]/tot:5.2f}  epi-waits-acc {s[3]/tot:5.2f}  cta_cycles/148={tot/148:9.0f}")
