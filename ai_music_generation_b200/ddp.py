"""Data-parallel wrapper for GPT (reference: torch DDP at nanoGPT/train.py:226-227, the
`model.require_backward_grad_sync` toggle at :341 and `raw_model = model.module` at :279).

One process per GPU (torchrun).  Gradients already live in one flat fp32 arena, so a bucket is a slice: no
flatten/copy kernels.  Buckets follow the order in which the backward plan completes layers (last block
first); each bucket's all-reduce (average) is enqueued on a side stream as soon as its last layer's wgrad
has been launched, overlapping NCCL over NVLink with the remaining backward.  The embedding / lm_head tensor
and the 1-D parameters finish last and form the final bucket.  `wait()` makes the compute stream wait for the
outstanding collectives (device-side; no host sync) before clip / AdamW.

NVLS mode (the default when the GPUs share a multicast-capable NVLink switch; `DDP(..., nvls=False)` or ABCGPT_DDP_NVLS=0 keeps
NCCL): the gradient arena lives in symmetric multicast memory and every bucket is exchanged by ONE kernel of ours — each rank
reduces its 1/world share through the switch (multimem.ld_reduce), multicasts the mean into every replica and, in the same
pass, the partial sums of squares that clip_grad_norm_ needs (csrc/nvls.cu, include/abcgpt.h abcgpt_nvls_allreduce_sumsq).
The kernel runs in 128-thread CTAs that share SMs with the backward's persistent GEMM CTAs instead of taking SMs away from
their static tile schedule (what an NCCL kernel does), and the separate norm pass over the arena disappears.
"""
from __future__ import annotations

import os
import warnings

import torch
import torch.distributed as dist

from . import ops


def plan_buckets(layer_ranges, head_range, tail_range, bucket_elems, extra_ranges=()):
    """Groups per-layer [lo, hi) element ranges of the flat gradient arena into all-reduce buckets.

    layer_ranges[i] is the contiguous range of block i's 2-D gradients; ranges are adjacent and ascending.
    `extra_ranges`: 2-D tensors registered after the last block (the hierarchical model's patch embedding).
    Returns [(trigger_layer, lo, hi)] in launch order (trigger_layer = the layer whose completion releases the
    bucket; -1 for the final bucket(s) released when the whole backward is done)."""
    buckets = []
    hi = None
    lo = None
    for li in range(len(layer_ranges) - 1, -1, -1):
        l_lo, l_hi = layer_ranges[li]
        if hi is None:
            hi = l_hi
        lo = l_lo
        if hi - lo >= bucket_elems or li == 0:
            buckets.append((li, lo, hi))
            hi = None
    for lo_, hi_ in (head_range, *extra_ranges, tail_range):
        if hi_ > lo_:
            buckets.append((-1, lo_, hi_))
    return buckets


def merge_final_buckets(buckets):
    """NVLS mode: the lowest layer group (trigger 0) joins the ranges released when the backward ends (trigger -1), and ranges that
    are adjacent in the arena (head | group, patch embedding | 1-D tail) become one range — fewer exposed launches, each of which
    sits between two device-side barriers.  The result still tiles exactly the same elements."""
    last = [b for b in buckets if b[0] <= 0]
    rest = [b for b in buckets if b[0] > 0]
    merged = []
    for _, lo, hi in sorted(last, key=lambda b: b[1]):
        if merged and merged[-1][2] == lo:
            merged[-1] = (-1, merged[-1][1], hi)
        else:
            merged.append((-1, lo, hi))
    return rest + merged


class GradSync:
    def __init__(self, grad_flat, layer_ranges, head_range, tail_range, process_group=None, bucket_mb=64.0,
                 extra_ranges=(), defer_final=False, nvls=None):
        self.grad = grad_flat
        self.nvls = nvls           # symmetric-memory state of the NVLS mode (see nvls_setup) or None: NCCL buckets
        self.norm_fresh = False    # NVLS: the partial-norm table describes the gradients currently in the arena
        self.group = process_group
        self.world = dist.get_world_size(process_group)
        self.buckets = plan_buckets(layer_ranges, head_range, tail_range, int(bucket_mb * 1024 * 1024 / 4), extra_ranges)
        # defer_final: gradients outside the block stack are still being produced when the stack's backward plan ends
        # (the patch embedding of the hierarchical model, computed by a later autograd node): the owner calls finalize()
        self.defer_final = defer_final
        self._by_trigger = {}
        for b in self.buckets:
            self._by_trigger.setdefault(b[0], []).append(b)
        self.cuda = grad_flat.is_cuda
        # high priority: the exchange kernels are tiny (NVLS) or latency-bound (NCCL) and should not queue behind compute CTAs
        self.comm_stream = torch.cuda.Stream(device=grad_flat.device, priority=-1 if nvls is not None else 0) if self.cuda else None
        self._pending = []
        self.launched = []  # (lo, hi) in launch order, for tests
        if nvls is not None:
            # every exchange costs a pair of device-side barriers, and the ones released at the END of the backward are exposed:
            # the lowest layer group joins the ranges around it (head | group | ... and patch embedding | 1-D tail are adjacent in
            # the arena), so the backward ends with one or two launches instead of four
            self.buckets = merge_final_buckets(self.buckets)
            self._by_trigger = {}
            for b in self.buckets:
                self._by_trigger.setdefault(b[0], []).append(b)
            # one table slot per (bucket, rank, block): many-layer models get fewer blocks per launch
            cap = nvls["table"].numel() // max(1, len(self.buckets) * self.world)
            nvls["bmax"] = max(1, min(296, cap))
            nvls["blocks"] = max(1, min(nvls["blocks"], nvls["bmax"]))

    def _launch(self, bucket):
        _, lo, hi = bucket
        view = self.grad[lo:hi]
        self.launched.append((lo, hi))
        if self.world == 1:
            return
        if self.nvls is not None:
            # NVLS, overlapped: the bucket's exchange runs on the communication stream as soon as the bucket's last wgrad has
            # been enqueued, in 128-thread CTAs that share SMs with the backward's persistent kernels (csrc/nvls.cu)
            ready = torch.cuda.Event()
            ready.record(torch.cuda.current_stream())
            with torch.cuda.stream(self.comm_stream):
                self.comm_stream.wait_event(ready)
                final = bucket[0] < 0   # released when the backward has ended: nothing left to disturb, full-size launch
                self._nvls_exchange(lo, hi, self.buckets.index(bucket), self.nvls["bmax"] if final else self.nvls["blocks"],
                                    512 if final else self.nvls["threads"])
            self.nvls["dirty"] = True
        elif self.cuda:
            ready = torch.cuda.Event()
            ready.record(torch.cuda.current_stream())
            with torch.cuda.stream(self.comm_stream):
                self.comm_stream.wait_event(ready)
                work = dist.all_reduce(view, op=dist.ReduceOp.AVG, group=self.group, async_op=True)
            self._pending.append(work)
        else:  # gloo on CPU (tests): no AVG reduction there
            dist.all_reduce(view, op=dist.ReduceOp.SUM, group=self.group)
            view.div_(self.world)

    def _nvls_exchange(self, lo, hi, slot, blocks, threads):
        """On the current stream: barrier (every rank has finished writing this range of its arena), the fused reduce +
        multicast + norm-partials kernel on this rank's share of the range, barrier (every share has landed in every replica)."""
        nv = self.nvls
        hdl = nv["hdl"]
        hdl.barrier(channel=0)
        ops.nvls_allreduce_sumsq(hdl.multicast_ptr + 4 * lo, hi - lo, hdl.rank, hdl.world_size,
                                 nv["thdl"].multicast_ptr + 4 * (slot * hdl.world_size + hdl.rank) * nv["bmax"], blocks, threads)
        hdl.barrier(channel=0)

    def layer_done(self, li):
        if self.nvls is not None and not self.nvls["overlap"]:
            return   # one exchange of the whole arena at the end of the backward (finalize)
        for b in self._by_trigger.get(li, ()):
            self._launch(b)

    def backward_done(self):
        if not self.defer_final:
            self.finalize()

    def finalize(self):
        """Releases the final bucket(s) and JOINS: the compute stream waits (device-side) for every outstanding collective.
        After `loss.backward()` returns, anything the caller enqueues on the compute stream — the reference loop's stock
        `torch.nn.utils.clip_grad_norm_(model.parameters(), ...)` (nanoGPT/train.py:350-352), `scaler.step`, a gradient
        read — therefore sees fully reduced gradients, exactly as with torch DDP.  Nothing else is queued behind the
        backward at this point, so the join costs no overlap."""
        if self.nvls is not None and not self.nvls["overlap"]:
            if self.world > 1:
                self._nvls_exchange(0, self.grad.numel(), 0, self.nvls["bmax"], 512)   # one launch, the GPU to itself
            self.launched.append((0, self.grad.numel()))
        else:
            for b in self._by_trigger.get(-1, ()):
                self._launch(b)
        self._join()
        if self.nvls is not None:
            self.nvls["version"] = self.grad._version
            self.norm_fresh = True

    def fused_sumsq(self, out):
        """NVLS mode: adds the squared norm of the exchanged gradients to out[0] from the partial table (no pass over the
        arena); False when the table does not describe the arena's current contents (then the caller runs its own pass)."""
        nv = self.nvls
        if nv is None or not self.norm_fresh or nv.get("version") != self.grad._version:
            return False
        # table layout [bucket][rank][bmax]; slots a launch did not use stay zero
        ops.sumsq_partials(nv["table"], (len(self.buckets) if nv["overlap"] else 1) * self.world * nv["bmax"], out)
        return True

    def _join(self):
        if self.nvls is not None:
            if self.nvls.get("dirty"):
                done = torch.cuda.Event()
                done.record(self.comm_stream)
                torch.cuda.current_stream().wait_event(done)
                self.nvls["dirty"] = False
            return
        for w in self._pending:
            w.wait()  # NCCL: the current stream waits for the collective; the host does not block
        self._pending = []

    def wait(self):
        self._join()
        self.launched = []


def nvls_requested(flag=None):
    """Default ("auto"): the NVLS exchange for gradient arenas of at least 128 MB whenever there is more than one rank (nvls_setup
    falls back to NCCL with a warning when the GPUs have no multicast memory); ABCGPT_DDP_NVLS=0 / 1 force NCCL / NVLS.  MEASURED (cfg3, one box each, profiles/r2b_nvls.md):
    8 GPUs 25.80 -> 25.15 / 25.25 ms per step, 2 GPUs 25.32 -> 25.03 ms."""
    if flag is None:
        e = os.environ.get("ABCGPT_DDP_NVLS", "auto")
        return "auto" if e == "auto" else e != "0"
    return bool(flag)


NVLS_AUTO_MIN_BYTES = 128 << 20   # "auto": arenas below this stay on NCCL (baby GPT, 43 MB, 2 GPUs: 2.67 ms NCCL vs 2.73 ms NVLS —
                                  # a handful of small exchanges, each between two device-side barriers, against one all-reduce)


def nvls_setup(m, process_group=None):
    """Moves the module's gradient arena into symmetric multicast memory (torch.distributed._symmetric_memory: allocation and
    handle exchange only) and allocates the partial-norm table.  Returns the state dict GradSync keeps, or None (with one
    warning) when the GPUs do not share a multicast-capable NVLink switch / the allocation fails: the caller falls back to NCCL."""
    a = m._arena
    try:
        import torch.distributed._symmetric_memory as symm_mem
        group = process_group if process_group is not None else dist.group.WORLD
        dev = a["flat"].device
        g = symm_mem.empty(a["total"], dtype=torch.float32, device=dev)
        hdl = symm_mem.rendezvous(g, group)
        table = symm_mem.empty(65536, dtype=torch.float32, device=dev)   # [buckets x world x blocks] partial sums of squares
        thdl = symm_mem.rendezvous(table, group)
        ok = torch.tensor([1 if (hdl.multicast_ptr and thdl.multicast_ptr and a["total"] % 4 == 0) else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=process_group)   # all ranks take the same path
        if int(ok.item()) == 0:
            raise RuntimeError("no multicast address for the symmetric allocation")
    except Exception as e:  # noqa: BLE001 - any failure here means "use NCCL"
        warnings.warn(f"NVLS gradient exchange unavailable ({type(e).__name__}: {e}); using NCCL all-reduce buckets")
        return None
    g.zero_()
    table.zero_()
    if a["grad"] is not None:
        g.copy_(a["grad"])
    a["grad"] = g
    for p, o in zip(a["params"], a["offs"]):   # existing .grad views follow the arena
        if p.grad is not None:
            p.grad = g[o:o + p.numel()].view(p.shape)
    m._bufs = {}   # recorded launch plans hold the old arena's pointers
    # overlap (default): bucket by bucket beside the backward, `blocks` CTAs of `threads` threads per launch (one 128-thread CTA per SM
    # fits next to a persistent GEMM CTA); the ranges released when the backward has ended go out in one full-size launch.
    # ABCGPT_NVLS_OVERLAP=0: one exchange of the whole arena after the backward.
    overlap = os.environ.get("ABCGPT_NVLS_OVERLAP", "1") != "0"
    return {"hdl": hdl, "thdl": thdl, "table": table, "overlap": overlap,
            "blocks": int(os.environ.get("ABCGPT_NVLS_BLOCKS", "148")), "threads": int(os.environ.get("ABCGPT_NVLS_THREADS", "128"))}


def attach_grad_sync(m, process_group=None, bucket_mb=64.0, defer_final=False, nvls=False):
    """Builds the GradSync of one GPT-shaped module over its flat gradient arena and stores it in m._grad_sync."""
    m._ensure_device_state()
    nv = None
    if nvls == "auto":
        nvls = m._arena["total"] * 4 >= NVLS_AUTO_MIN_BYTES
    if nvls and m._arena["flat"].is_cuda and dist.get_world_size(process_group) > 1:
        nv = nvls_setup(m, process_group)
    if nv is not None:   # per-layer buckets: the last exchange (the exposed one) stays short; measured 25.15 -> 25.03 ms at N = 2
        bucket_mb = min(bucket_mb, float(os.environ.get("ABCGPT_NVLS_BUCKET_MB", "25")))
    a = m._arena
    names, offs, params = a["names"], a["offs"], a["params"]
    end = {n: o + ((p.numel() + 7) // 8) * 8 for n, o, p in zip(names, offs, params)}
    start = dict(zip(names, offs))
    layer_ranges = []
    for i in range(m.config.n_layer):
        pre = f"transformer.h.{i}."
        layer_ranges.append((start[pre + "attn.c_attn.weight"], end[pre + "mlp.c_proj.weight"]))
    head = (0, layer_ranges[0][0]) if layer_ranges else (0, a["n_decay"])
    extra = [(layer_ranges[-1][1], a["n_decay"])] if layer_ranges else []
    tail = (a["n_decay"], a["total"])
    m._grad_sync = GradSync(a["grad"], layer_ranges, head, tail, process_group, bucket_mb, extra_ranges=extra,
                            defer_final=defer_final, nvls=nv)
    return m._grad_sync


class DDP(torch.nn.Module):
    """Thin container with the two attributes the reference's training loop touches."""

    def __init__(self, module, device_ids=None, process_group=None, bucket_mb=64.0, nvls=None):
        super().__init__()
        self.module = module
        self._process_group = process_group
        self._bucket_mb = bucket_mb
        self._nvls = nvls_requested(nvls)
        self._sync_for = None
        if dist.is_initialized() and dist.get_world_size(process_group) > 1:
            flat = module._arena["flat"]
            dist.broadcast(flat, src=0, group=process_group)  # same start on every rank, like DDP's constructor
            module._shadow_fresh = False

    @property
    def require_backward_grad_sync(self):
        return self.module.require_backward_grad_sync

    @require_backward_grad_sync.setter
    def require_backward_grad_sync(self, value):
        self.module.require_backward_grad_sync = bool(value)

    def _ensure_sync(self):
        m = self.module
        m._ensure_device_state()
        if self._sync_for == m._arena["grad"].data_ptr():
            return
        attach_grad_sync(m, self._process_group, self._bucket_mb, nvls=self._nvls)
        self._sync_for = m._arena["grad"].data_ptr()   # (the NVLS mode replaces the arena)

    def forward(self, *args, **kwargs):
        if dist.is_initialized():
            self._ensure_sync()
        return self.module(*args, **kwargs)

    def parameters(self, recurse=True):
        return self.module.parameters(recurse)

    def clip_grad_norm_(self, max_norm):
        return self.module.clip_grad_norm_(max_norm)


class TunesFormerDDP(torch.nn.Module):
    """Data parallelism for the hierarchical model (tunesformer.TunesFormerShaped; the reference trains it under
    torch DataParallel / DDP, tunesformer/train.py): one GradSync per decoder arena.  The character-level decoder's
    backward runs first and releases its buckets layer by layer, then the patch-level stack's; the patch embedding's
    gradient is produced by a later autograd node, so that arena's final buckets are released from there
    (`finalize()`).  clip_grad_norm_ / the optimizer wait on both."""

    def __init__(self, module, process_group=None, bucket_mb=64.0):
        super().__init__()
        self.module = module
        self._process_group = process_group
        self._bucket_mb = bucket_mb
        self._sync_for = None
        if dist.is_initialized() and dist.get_world_size(process_group) > 1:
            for dec in (module.patch_level_decoder, module.char_level_decoder):
                dist.broadcast(dec._arena["flat"], src=0, group=process_group)
                dec._shadow_fresh = False

    @property
    def require_backward_grad_sync(self):
        return self.module.char_level_decoder.require_backward_grad_sync

    @require_backward_grad_sync.setter
    def require_backward_grad_sync(self, value):
        for dec in (self.module.patch_level_decoder, self.module.char_level_decoder):
            dec.require_backward_grad_sync = bool(value)

    def _ensure_sync(self):
        p, c = self.module.patch_level_decoder, self.module.char_level_decoder
        p._ensure_device_state()
        c._ensure_device_state()
        key = (p._arena["grad"].data_ptr(), c._arena["grad"].data_ptr())
        if self._sync_for == key:
            return
        attach_grad_sync(c, self._process_group, self._bucket_mb)
        attach_grad_sync(p, self._process_group, self._bucket_mb, defer_final=True)
        self._sync_for = key

    def forward(self, *args, **kwargs):
        if dist.is_initialized():
            self._ensure_sync()
        return self.module(*args, **kwargs)

    def parameters(self, recurse=True):
        return self.module.parameters(recurse)

    def clip_grad_norm_(self, max_norm):
        return self.module.clip_grad_norm_(max_norm)
