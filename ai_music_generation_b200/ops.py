"""Tensor-level wrappers over the C ABI: torch supplies device memory and the stream, nothing else.

Every function enqueues hand-written sm_100a kernels on torch's current CUDA stream through libabcgpt.so and
raises AbcgptError on failure.  No function here computes anything with torch ops.
"""
from __future__ import annotations

import torch

from . import _C
from ._C import ACT_TANH, EPI_BF16, EPI_DGELU, EPI_F32, EPI_F32_RED, EPI_GELU, EPI_RESID  # noqa: F401


LAUNCHES = 0      # kernels of libabcgpt.so enqueued so far (bench.py reports the delta over its timed region)
CALLS = 0         # calls into libabcgpt.so that enqueue work (a compiled replay of a whole launch list counts once)
_PROFILE = None   # optional list collecting (name, meta, start_event, end_event) per C-ABI call


def set_profile(sink):
    """sink: None or a list; when set, every call is bracketed by CUDA events on the launching stream."""
    global _PROFILE
    _PROFILE = sink


_RECORD = None    # launch-plan recording: list of (name, nkernels, fn, args) / ("py", callable)


def begin_record():
    """Start recording every C-ABI call (they still execute).  All pointers of a plan are static (arena + per-shape buffers),
    so a recorded plan can be replayed with ~1 us of Python per launch instead of re-deriving every argument."""
    global _RECORD
    _RECORD = []


def end_record():
    global _RECORD
    plan, _RECORD = _RECORD, None
    return plan


_KEYED = ("embed_fwd", "embed_bwd", "layernorm_fwd_resid", "layernorm_bwd", "attn_fwd", "attn_bwd", "gemm")


def key_patches(plan, keys):
    """Dropout sites of a recorded plan: [(entry index, site)] for every launch that carries a dropout key (their C signatures
    all end `..., dropout_p, dropout_key, stream`).  The keys are the only arguments of a training plan that change from step to
    step, so a plan recorded with one step's keys is replayed with the next step's (`replay(plan, patches, keys)`).  Returns None
    when the sites cannot be told apart (two sites with the same 32-bit key)."""
    if len(set(keys)) != len(keys):
        return None
    site_of = {k: i for i, k in enumerate(keys)}
    out = []
    for i, e in enumerate(plan):
        if e[0] in _KEYED and float(e[3][-3]) > 0.0:
            site = site_of.get(int(e[3][-2]))
            if site is None:
                return None
            plan[i] = (e[0], e[1], e[2], list(e[3]), e[4])
            out.append((i, site))
    return out


def set_pdl(on):
    """Programmatic dependent launch for the launches that follow (include/abcgpt.h: abcgpt_set_pdl)."""
    _C.lib().abcgpt_set_pdl(1 if on else 0)


_SIDE = {}


def side_stream():
    """The second stream of the current device for kernels that are independent of the main chain (weight-gradient GEMMs)."""
    dev = torch.cuda.current_device()
    st = _SIDE.get(dev)
    if st is None:
        st = _SIDE[dev] = torch.cuda.Stream(device=dev)
    return st


def profiling():
    return _PROFILE is not None


def event_record(slot, stream=None):
    """include/abcgpt.h abcgpt_event_record: mark the work enqueued so far on `stream` (default: the current one) under `slot`."""
    _call("event_record", 0, (slot,), _C.lib().abcgpt_event_record, int(slot), _stream() if stream is None else stream.cuda_stream)


def event_wait(slot, stream=None):
    """abcgpt_event_wait: `stream` (default: the current one) waits on the device for the latest mark of `slot`."""
    _call("event_wait", 0, (slot,), _C.lib().abcgpt_event_wait, int(slot), _stream() if stream is None else stream.cuda_stream)


def record_callback(fn):
    """Interleave a Python callback (e.g. DDP bucket launch) with the recorded launches; runs now and on every replay."""
    global _RECORD
    rec = _RECORD
    if rec is not None:
        rec.append(("py", fn))
    _RECORD = None   # launches made BY the callback belong to the callback (it runs again on every replay), not to the plan
    try:
        fn()
    finally:
        _RECORD = rec


def replay(plan, patches=None, keys=None):
    global LAUNCHES, CALLS
    if patches:
        for i, site in patches:
            plan[i][3][-2] = keys[site]
    if _PROFILE is not None:  # instrumented pass: fall back to event-bracketed calls
        for e in plan:
            if e[0] == "py":
                e[1]()
            else:
                _call(e[0], e[1], e[4], e[2], *e[3])
        return
    for e in plan:
        if e[0] == "py":
            e[1]()
            continue
        LAUNCHES += e[1]
        CALLS += 1
        rc = e[2](*e[3])
        if rc != 0:
            _C.check(rc, e[0])


def plan_deltas(plan_a, plan_b):
    """Per-launch argument differences between two recorded plans of the same structure (None if they do not match):
    [(patch list [(arg index, delta)])].  Decode steps at consecutive positions differ only in arguments that are affine in
    the position (cache row pointers, token column pointers, the key count), so one recorded step can be replayed at any
    position by adding k * delta."""
    if len(plan_a) != len(plan_b):
        return None
    out = []
    for ea, eb in zip(plan_a, plan_b):
        if ea[0] == "py" or eb[0] == "py" or ea[0] != eb[0] or ea[2] is not eb[2] or len(ea[3]) != len(eb[3]):
            return None
        patches = []
        for i, (x, y) in enumerate(zip(ea[3], eb[3])):
            if x == y:
                continue
            if not (isinstance(x, int) and isinstance(y, int)):
                return None
            patches.append((i, y - x))
        out.append(patches)
    return out


def compile_affine(plan, deltas):
    """Pack a recorded plan + its per-position argument deltas into the int64 program abcgpt_replay executes in C (one ctypes
    call per decode step instead of ~90).  Returns (program array, words, launches) or None if a call cannot be encoded."""
    import ctypes
    import struct
    words = []
    launches = 0
    for e, patches in zip(plan, deltas):
        fid = _C.FN_IDS.get(getattr(e[2], "__name__", ""))
        if fid is None:
            return None
        d = dict(patches)
        words += [fid, len(e[3])]
        for i, a in enumerate(e[3]):
            if isinstance(a, float):
                words += [struct.unpack("<q", struct.pack("<d", a))[0], 0]
            elif a is None:
                words += [0, 0]
            else:
                v = int(a)
                if v >= 1 << 63:
                    v -= 1 << 64
                words += [v, int(d.get(i, 0))]
        launches += e[1]
    arr = (ctypes.c_int64 * len(words))(*words)
    return arr, len(words), launches


def replay_compiled(prog, k):
    global LAUNCHES, CALLS
    arr, n, launches = prog
    LAUNCHES += launches
    CALLS += 1
    rc = _C.lib().abcgpt_replay(arr, n, k)
    if rc != 0:
        _C.check(rc, "abcgpt_replay")


def replay_affine(plan, deltas, k):
    """Replay `plan` with every patched argument advanced by k * delta (see plan_deltas)."""
    global LAUNCHES, CALLS
    if _PROFILE is not None or _RECORD is not None:
        raise _C.AbcgptError("replay_affine: not available while profiling / recording")
    for e, patches in zip(plan, deltas):
        LAUNCHES += e[1]
        CALLS += 1
        if patches:
            args = list(e[3])
            for i, d in patches:
                args[i] += k * d
            rc = e[2](*args)
        else:
            rc = e[2](*e[3])
        if rc != 0:
            _C.check(rc, e[0])


def _call(name, nkernels, meta, fn, *args):
    global LAUNCHES, CALLS
    LAUNCHES += nkernels
    CALLS += 1
    if _RECORD is not None:
        _RECORD.append((name, nkernels, fn, args, meta))
    if _PROFILE is None:
        rc = fn(*args)
    else:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = fn(*args)
        e1.record()
        _PROFILE.append((name, meta, e0, e1))
    if rc != 0:
        _C.check(rc, name)


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _chk(t, dtype, name):
    if not t.is_cuda:
        raise _C.AbcgptError(f"{name}: expected a CUDA tensor (there is no CPU fallback)")
    if t.dtype != dtype:
        raise _C.AbcgptError(f"{name}: expected dtype {dtype}, got {t.dtype}")


def _rowmajor_ld(t, name):
    if t.dim() != 2 or t.stride(1) != 1:
        raise _C.AbcgptError(f"{name}: expected a 2-D tensor with unit inner stride, got strides {t.stride()}")
    return t.stride(0)


def gemm(a, b, *, a_mn=False, b_mn=False, M=None, N=None, K=None, epilogue=EPI_BF16, out=None, out2=None, aux=None,
         bias=None, tile_n=0, splits=0, drop_p=0.0, drop_key=0, head_stride=0):
    """out[M,N] = sum_k A[m,k] B[n,k] (bf16 in, fp32 accumulate on tcgen05).

    a: [M,K] (a_mn=False) or stored [K,M] (a_mn=True); b: [N,K] or stored [K,N].
    head_stride (EPI_BF16 only): column c of output row m is stored at out[m, 0] + (c // 64) * head_stride + c % 64 — the
    head-major KV cache of the decode path (`out` is then the [M, 64] view of the first head at the current position)."""
    _chk(a, torch.bfloat16, "gemm a")
    _chk(b, torch.bfloat16, "gemm b")
    lda, ldb = _rowmajor_ld(a, "gemm a"), _rowmajor_ld(b, "gemm b")
    Ma, Ka = (a.shape[1], a.shape[0]) if a_mn else (a.shape[0], a.shape[1])
    Nb, Kb = (b.shape[1], b.shape[0]) if b_mn else (b.shape[0], b.shape[1])
    M = Ma if M is None else M
    N = Nb if N is None else N
    K = Ka if K is None else K
    if Ka != Kb and (K is None):
        raise _C.AbcgptError(f"gemm: contraction mismatch {Ka} vs {Kb}")
    ldc = _rowmajor_ld(out, "gemm out")
    ldc2 = _rowmajor_ld(out2, "gemm out2") if out2 is not None else int(head_stride)
    ldaux = _rowmajor_ld(aux, "gemm aux") if aux is not None else 0
    if bias is not None:
        _chk(bias, torch.float32, "gemm bias")
    _call("gemm", 1, (M, N, K, int(a_mn), int(b_mn), epilogue), _C.lib().abcgpt_gemm_bf16, a.data_ptr(), int(a_mn), lda,
          b.data_ptr(), int(b_mn), ldb, M, N, K, epilogue, out.data_ptr(), ldc, _ptr(out2), ldc2, _ptr(aux), ldaux,
          _ptr(bias), tile_n, splits, drop_p, drop_key, _stream())
    return out


def add_pos(e, wpe, x, T):
    """x[m] = e[m] + wpe[m % T] (fp32): a decoder fed with embeddings from another network."""
    _chk(e, torch.float32, "add_pos e")
    M, C = x.shape
    _call("add_pos", 1, (M, C), _C.lib().abcgpt_add_pos, e.data_ptr(), wpe.data_ptr(), x.data_ptr(), M, T, C, _stream())


def set_first_pos(first, wpe, x, T):
    """x[b, 0] = first[b] + wpe[0]: the encoded bar patch replaces the first character embedding."""
    _chk(first, torch.float32, "set_first_pos first")
    Bn, C = first.shape
    _call("set_first_pos", 1, (Bn, C), _C.lib().abcgpt_set_first_pos, first.data_ptr(), wpe.data_ptr(), x.data_ptr(), Bn, T, C,
          _stream())


def pos_bwd(dx, dwpe, T):
    M, C = dx.shape
    _call("pos_bwd", 1, (M, C), _C.lib().abcgpt_pos_bwd, dx.data_ptr(), dwpe.data_ptr(), M, T, C, _stream())


def onehot_bf16(tok, out, V):
    """out[m, s * V + tok[m, s]] = 1 (bf16), everything else 0: the rows TunesFormer's patch embedding Linear sees."""
    _chk(tok, torch.int64, "onehot tok")
    M, S = tok.shape
    _call("onehot", 1, (M, S, V), _C.lib().abcgpt_onehot_bf16, tok.data_ptr(), out.data_ptr(), M, S, V, _stream())


def embed_fwd(idx, wte, wpe, x, T, drop_p=0.0, drop_key=0):
    _chk(idx, torch.int64, "embed idx")
    M = idx.numel()
    V, C = wte.shape
    _call("embed_fwd", 1, (M, C), _C.lib().abcgpt_embed_fwd, idx.data_ptr(), wte.data_ptr(), wpe.data_ptr(), x.data_ptr(),
          M, T, C, V, drop_p, drop_key, _stream())
    return x


def embed_bwd(idx, dx, dwte, dwpe, T, drop_p=0.0, drop_key=0):
    M = idx.numel()
    V, C = dwte.shape
    _call("embed_bwd", 2, (M, C), _C.lib().abcgpt_embed_bwd, idx.data_ptr(), dx.data_ptr(), dwte.data_ptr(),
          dwpe.data_ptr(), M, T, C, V, drop_p, drop_key, _stream())


def layernorm_fwd(x, weight, bias, y_bf16, mean, rstd, y_f32=None):
    _chk(x, torch.float32, "layernorm x")
    M, C = x.shape
    _call("layernorm_fwd", 1, (M, C), _C.lib().abcgpt_layernorm_fwd, x.data_ptr(), weight.data_ptr(), _ptr(bias),
          _ptr(y_bf16), _ptr(y_f32), _ptr(mean), _ptr(rstd), M, C, _stream())


def layernorm_fwd_resid(x_in, branch_bf16, x_out, weight, bias, y_bf16, mean, rstd, drop_p=0.0, drop_key=0):
    """x_out = x_in + [dropout](branch), y = LN(x_out) in one pass (include/abcgpt.h: abcgpt_layernorm_fwd_resid)."""
    _chk(x_in, torch.float32, "layernorm x_in")
    _chk(branch_bf16, torch.bfloat16, "layernorm branch")
    M, C = x_in.shape
    _call("layernorm_fwd_resid", 1, (M, C), _C.lib().abcgpt_layernorm_fwd_resid, x_in.data_ptr(), branch_bf16.data_ptr(),
          x_out.data_ptr(), weight.data_ptr(), _ptr(bias), y_bf16.data_ptr(), _ptr(mean), _ptr(rstd), M, C, drop_p, drop_key,
          _stream())


def layernorm_bwd(dy_bf16, x, weight, mean, rstd, dresid_in, dx_out, dx_bf16, dweight, dbias, drop_p=0.0, drop_key=0):
    M, C = x.shape
    _call("layernorm_bwd", 1, (M, C), _C.lib().abcgpt_layernorm_bwd, dy_bf16.data_ptr(), x.data_ptr(), weight.data_ptr(),
          mean.data_ptr(), rstd.data_ptr(), _ptr(dresid_in), dx_out.data_ptr(), _ptr(dx_bf16), _ptr(dweight),
          _ptr(dbias), M, C, drop_p, drop_key, _stream())


def attn_fwd(qkv, out, lse, B, T, H, drop_p=0.0, drop_key=0, head_size=64):
    """Causal attention over the packed [B*T, 3C] qkv buffer, C = H * head_size.  head_size 64 runs the tuned kernels of
    csrc/attn.cu; 32 and 128 those of csrc/attn_hd.cu (abcgpt_attn_fwd_hd), recorded under the same name so that a launch
    plan patches their dropout keys like any other attention launch."""
    _chk(qkv, torch.bfloat16, "attn qkv")
    if head_size == 64:
        _call("attn_fwd", 1, (B, T, H), _C.lib().abcgpt_attn_fwd, qkv.data_ptr(), out.data_ptr(), lse.data_ptr(), B, T, H,
              drop_p, drop_key, _stream())
    else:
        _call("attn_fwd", 1, (B, T, H, head_size), _C.lib().abcgpt_attn_fwd_hd, qkv.data_ptr(), out.data_ptr(), lse.data_ptr(),
              B, T, H, int(head_size), drop_p, drop_key, _stream())


def attn_bwd(qkv, out, dout, lse, delta, dqkv, B, T, H, drop_p=0.0, drop_key=0, head_size=64):
    if head_size == 64:
        _call("attn_bwd", 3, (B, T, H), _C.lib().abcgpt_attn_bwd, qkv.data_ptr(), out.data_ptr(), dout.data_ptr(),
              lse.data_ptr(), delta.data_ptr(), dqkv.data_ptr(), B, T, H, drop_p, drop_key, _stream())
    else:
        _call("attn_bwd", 3, (B, T, H, head_size), _C.lib().abcgpt_attn_bwd_hd, qkv.data_ptr(), out.data_ptr(), dout.data_ptr(),
              lse.data_ptr(), delta.data_ptr(), dqkv.data_ptr(), B, T, H, int(head_size), drop_p, drop_key, _stream())


def ce_fwd(logits, targets, row_loss, sum_count, loss, V):
    _chk(logits, torch.bfloat16, "ce logits")
    _chk(targets, torch.int64, "ce targets")
    M, ldl = logits.shape[0], logits.stride(0)
    L = _C.lib()
    _call("ce_fwd", 1, (M, V), L.abcgpt_ce_fwd, logits.data_ptr(), ldl, targets.data_ptr(), row_loss.data_ptr(), M, V,
          _stream())
    _call("ce_finalize", 1, (M,), L.abcgpt_ce_finalize, row_loss.data_ptr(), targets.data_ptr(), M, sum_count.data_ptr(),
          _ptr(loss), _stream())


def ce_bwd(logits, targets, sum_count, grad_loss, dlogits, V):
    M, ldl = logits.shape[0], logits.stride(0)
    _call("ce_bwd", 1, (M, V), _C.lib().abcgpt_ce_bwd, logits.data_ptr(), ldl, targets.data_ptr(), sum_count.data_ptr(),
          grad_loss.data_ptr(), dlogits.data_ptr(), M, V, _stream())


_SUMSQ_WS = {}


def sumsq(g, out):
    ws = _SUMSQ_WS.get(g.device)
    if ws is None:
        ws = _SUMSQ_WS[g.device] = torch.empty(1024, device=g.device, dtype=torch.float32)
    _call("sumsq", 2, (g.numel(),), _C.lib().abcgpt_sumsq, g.data_ptr(), g.numel(), out.data_ptr(), ws.data_ptr(), _stream())


def adamw(p, g, m, v, shadow, *, lr, beta1, beta2, eps, weight_decay, step, sumsq=None, max_norm=0.0):
    _call("adamw", 1, (p.numel(),), _C.lib().abcgpt_adamw, p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(),
          _ptr(shadow), p.numel(), lr, beta1, beta2, eps, weight_decay, step, _ptr(sumsq), max_norm, _stream())


def cast_bf16(x, y):
    _call("cast_bf16", 1, (x.numel(),), _C.lib().abcgpt_cast_f32_to_bf16, x.data_ptr(), y.data_ptr(), x.numel(), _stream())


def argmax(logits, V, out, out_stride=1):
    B, ldl = logits.shape[0], logits.stride(0)
    _call("argmax", 1, (B, V), _C.lib().abcgpt_argmax, logits.data_ptr(), ldl, V, out.data_ptr(), out_stride, B, _stream())


def sample_topk(logits, V, out, temperature, top_k, seed, counter, out_stride=1):
    """One multinomial draw per row from softmax(top-k(logits / temperature)) (include/abcgpt.h: abcgpt_sample_topk).
    seed: uint64 device scalar (int64 tensor of one element); counter: the decode position."""
    _chk(logits, torch.bfloat16, "sample logits")
    B, ldl = logits.shape[0], logits.stride(0)
    _call("sample_topk", 1, (B, V), _C.lib().abcgpt_sample_topk, logits.data_ptr(), ldl, V, float(temperature),
          int(top_k) if top_k is not None else 0, seed.data_ptr(), int(counter), out.data_ptr(), out_stride, B, _stream())


def sample_top_p(logits, V, out, top_p, top_k, temperature, seed, counter_base, counter, row_id=None, out_stride=1):
    """Nucleus, then top-k, then temperature, one draw per row (include/abcgpt.h: abcgpt_sample_top_p).  seed / counter_base:
    int64 device scalars; counter: the decode position; row_id: optional int64 [B] device tensor naming each row's stream."""
    _chk(logits, torch.bfloat16, "sample logits")
    B, ldl = logits.shape[0], logits.stride(0)
    _call("sample_top_p", 1, (B, V), _C.lib().abcgpt_sample_top_p, logits.data_ptr(), ldl, V, float(top_p), int(top_k),
          float(temperature), seed.data_ptr(), counter_base.data_ptr(), int(counter), _ptr(row_id), out.data_ptr(), out_stride, B,
          _stream())


def nvls_allreduce_sumsq(grad_mc_ptr, n, rank, world, partials_mc_ptr, blocks_per_rank, threads=512):
    """include/abcgpt.h abcgpt_nvls_allreduce_sumsq: mean of the replicas' gradient arenas + norm partials, over multicast memory."""
    _call("nvls_allreduce_sumsq", 1, (n, world), _C.lib().abcgpt_nvls_allreduce_sumsq, int(grad_mc_ptr), int(n), int(rank), int(world),
          1.0 / world, int(partials_mc_ptr), int(blocks_per_rank), int(threads), _stream())


def set_dynamic_tiles(on):
    """include/abcgpt.h abcgpt_set_dynamic_tiles: ticket-based tile scheduler for the pair GEMM launches that follow."""
    _C.lib().abcgpt_set_dynamic_tiles(1 if on else 0)


def sumsq_partials(partials, nparts, out):
    _call("sumsq_partials", 1, (nparts,), _C.lib().abcgpt_sumsq_partials, partials.data_ptr(), int(nparts), out.data_ptr(), _stream())


def colsum_bf16(dy, out):
    M, N = dy.shape
    _call("colsum_bf16", 1, (M, N), _C.lib().abcgpt_colsum_bf16, dy.data_ptr(), dy.stride(0), M, N, out.data_ptr(), _stream())


def attn_decode(cache, out, B, Tmax, n_keys, H):
    _call("attn_decode", 1, (B, n_keys, H), _C.lib().abcgpt_attn_decode, cache.data_ptr(), out.data_ptr(), B, Tmax, n_keys, H,
          _stream())


def attn_decode_hd(qkv_row, cache, out, B, Tmax, t, H, head_size):
    """Decode position t for head sizes 32 / 128 (include/abcgpt.h abcgpt_attn_decode_hd): appends k, v of qkv_row [B, 3C] to the
    head-major cache [B, 2H, Tmax, head_size] and attends over its rows [0, t]; out [B, C]."""
    _call("attn_decode_hd", 1, (B, t + 1, H, head_size), _C.lib().abcgpt_attn_decode_hd, qkv_row.data_ptr(), cache.data_ptr(),
          out.data_ptr(), B, Tmax, t, H, int(head_size), _stream())


def sample_batch(data, ix, x, y):
    B, T = x.shape
    _call("sample_batch", 1, (B, T), _C.lib().abcgpt_sample_batch, data.data_ptr(), data.element_size(), data.numel(),
          ix.data_ptr(), x.data_ptr(), y.data_ptr(), B, T, _stream())
