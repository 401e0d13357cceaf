"""Fused Adam for the scene pipeline (reference: ``torch.optim.Adam(self.parameters(), lr)`` at
roadmap_bce_v2.py:155 / autoencoder.py:120, stepped by Lightning after ddp's gradient all-reduce).

One process per GPU.  With world size 1 every tensor is updated by one ``dd_adam_step`` launch; with
``overlap_backward=True`` the wide FC weights instead take their step inside the backward pass, in the same kernel that
computes their layer's input gradient (``dd_linear_bwd_adam``).
With world size N the parameters are *sharded across ranks for the update only*: gradient and
weight replicas live in one symmetric-memory buffer per rank
(``torch.distributed._symmetric_memory``: every replica is peer-mapped into every process, plus an
NVLink multicast mapping where the fabric has one), and ``dd_adam_step_sharded`` does reduce + Adam
+ all-gather in ONE kernel (csrc/adam.cu): 1/N of the optimizer state and of the optimizer's HBM
traffic per GPU, and no NCCL kernel in the step.

* The wide FC weights (>= ``shard_min_numel`` elements; > 99.9 % of the bytes) each own a region;
  ``ops.linear``'s weight-gradient kernel writes straight into the gradient replica (``p.grad`` is a
  persistent view that every backward pass OVERWRITES; ``zero_grad`` leaves it in place).  With
  ``overlap_backward=True`` their update is launched from the backward pass itself, as soon as the
  gradient is written, on a side stream with one small CTA per SM that co-resides with the
  persistent conv kernels of the remaining backward pass; ``step()`` joins it.
* All other tensors share one flat region: their gradients are gathered into it by one multi-tensor
  copy and updated by one sharded launch in ``step()``.

``state_dict()`` / ``load_state_dict()`` speak torch.optim.Adam's layout (per-parameter ``step`` / ``exp_avg`` /
``exp_avg_sq`` of the parameter's shape) at every world size: the moment shards live in a second symmetric buffer, so
the rank that writes a checkpoint (rank 0 under Lightning) assembles the full moments from its peers' shards without a
collective, and every rank re-slices its own shard on load -- a checkpoint moves between world sizes and to / from
torch.optim.Adam.

Gradient accumulation (``accumulate_grad_batches=k``, Lightning's flag of the same name): a *window* is the k backward
passes between two ``step()`` calls.  The wide weights' gradients add up within a window exactly as autograd adds them
(``dd_linear_wgrad_acc``: the first pass of a window overwrites, later passes add), and their Adam step runs once per
window -- inside the window's last backward pass where it can: world size N launches the sharded update from pass k,
world size 1 with ``overlap_backward=True`` runs ``dd_linear_bwd_adam_acc`` (step folded into the backward pass, 28 bytes
per parameter) on pass k, from a persistent gradient buffer per wide weight that holds passes 1 .. k-1.  A ``step()``
after fewer than k passes updates from the gradients gathered so far; ``zero_grad()`` discards an unfinished window; a
(k+1)-th pass without a ``step()`` is refused.  With ``overlap_backward=False`` at world size 1 the wide weights' gradients
go through autograd, which accumulates them itself.

Gradient clipping (``gradient_clip_val=c``, Lightning's flag of the same name; world size 1): the step applies
``torch.nn.utils.clip_grad_norm_(params, c)`` to the gradients it is about to apply -- every group, the window's accumulated
gradients -- before Adam.  The norm and the coefficient stay on the device (``dd_grad_sumsq``, then ``dd_adam_step_clipped``
per tensor), so the step has no host sync; ``last_grad_norm`` is the pre-clip total norm, as ``clip_grad_norm_`` returns it.
Clipping needs every gradient before any update, so under it the wide weights' step does not run inside the backward pass:
their gradients are written (or accumulated) and step() applies them.

Gradient norms (``track_grad_norm=2``, Lightning's flag of the same name): ``grad_norms()`` returns the L2 norm of every
gradient the window's step applies -- the accumulated window gradient, the rank mean at world size N, before any clipping --
as 0-dim fp32 device tensors, and their total, without a host sync.  The wide weights' sums of squares come from the kernels
that step them (``dd_linear_bwd_adam_sumsq``, ``dd_adam_step_sharded_sumsq``: at world size N each rank sums its shard and
every rank adds the N shard sums in rank order, so every rank holds the same bits); the stored gradients go through
``dd_grad_sumsq_each`` (``_replicas`` for the data-parallel flat bucket).  Tracking never changes an update.

Semantics are torch.optim.Adam's (amsgrad off, L2 weight decay); ``param_groups[i]['lr']`` is read
every step, so ``ReduceLROnPlateau`` (roadmap_bce_v2.py:156) works unchanged; tensors whose
gradient is ``None`` are skipped (a partly frozen flat bucket is updated per tensor on every replica).
"""
from __future__ import annotations

import ctypes
import math
import warnings
import weakref

import torch
import torch.distributed as dist

from . import _lib
from ._lib import call, stream_ptr

_ALIGN = 64          # elements: every tensor of the flat region starts on a 256-byte boundary


def shard_bounds(numel: int, world: int, rank: int):
    """Elements [lo, hi) of a flat tensor that ``rank`` updates: equal shards of 4-element (16 B)
    granules, the last rank takes the remainder granules.  numel must be a multiple of 4."""
    granules = numel // 4
    per = granules // world
    lo = rank * per
    hi = granules if rank == world - 1 else lo + per
    return 4 * lo, 4 * hi


def accumulation_factor(accumulate_grad_batches, epoch: int = 0) -> int:
    """The number of backward passes per optimizer step: an int, or Lightning's ``{epoch: factor}`` schedule (the factor
    of the largest epoch key <= ``epoch``; 1 before the first key)."""
    k = accumulate_grad_batches
    if isinstance(k, dict):
        k = next((k[e] for e in sorted(k, reverse=True) if epoch >= e), 1)
    if isinstance(k, bool) or int(k) != k or int(k) < 1:
        raise ValueError(f"accumulate_grad_batches must be a positive integer, got {k!r}")
    return int(k)


_NO_SHARDED_CLIP = ("FusedAdam: gradient_clip_val is supported at world size 1; the data-parallel form has no clipping yet "
                    "(its norm must be that of the rank-averaged gradient)")


def gradient_clip_value(c) -> float:
    """Lightning's ``gradient_clip_val``: the max_norm of clip_grad_norm_, 0.0 (or None) for off."""
    if c is None:
        return 0.0
    if isinstance(c, bool) or not isinstance(c, (int, float)) or not math.isfinite(c) or c < 0:
        raise ValueError(f"gradient_clip_val must be a finite number >= 0 (0 = off), got {c!r}")
    return float(c)


def track_grad_norm_value(t) -> bool:
    """Lightning's ``track_grad_norm``: -1, 0 or None for off; FusedAdam tracks the 2-norm only (2 or 2.0)."""
    if t is None or (not isinstance(t, bool) and isinstance(t, (int, float)) and t in (-1, 0)):
        return False
    if not isinstance(t, bool) and isinstance(t, (int, float)) and t == 2:
        return True
    raise ValueError(f"track_grad_norm: FusedAdam tracks the 2-norm only (track_grad_norm=2; -1, 0 or None for off), got {t!r}")


def flat_layout(numels, align: int = _ALIGN):
    """Offsets of tensors packed into one flat region (each start aligned) and the region's length."""
    offs, off = [], 0
    for n in numels:
        offs.append(off)
        off += -(-n // align) * align
    return offs, off


class FusedAdam(torch.optim.Optimizer):
    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, process_group=None,
                 shard_min_numel: int = 1 << 20, multicast: bool | None = None, broadcast_init: bool = True,
                 overlap_backward: bool = False, fuse_into_backward: bool = False, defer_join: bool = True,
                 accumulate_grad_batches=1, gradient_clip_val=0.0, track_grad_norm=-1):
        if lr < 0 or eps < 0 or not (0 <= betas[0] < 1) or not (0 <= betas[1] < 1) or weight_decay < 0:
            raise ValueError("invalid Adam hyper-parameters")
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))
        accumulation_factor(accumulate_grad_batches)          # validates an int (a schedule is checked per window)
        # backward passes per step: an int, or a {epoch: factor} schedule read at the first backward pass of each window
        # against self.current_epoch() (make_adam: the module's current_epoch); may be changed between steps
        self.accumulate_grad_batches = accumulate_grad_batches
        self.current_epoch = lambda: 0
        # last_grad_norm: the last clipped step's total norm, a 0-dim fp32 tensor on the device (None before)
        self._clip_val = gradient_clip_value(gradient_clip_val)
        self.last_grad_norm = None
        self._clip_ws = None        # dd_grad_sumsq's workspace (zeroed once, self-resetting)
        # gradient norms (grad_norms()): the window's fp64 sums of squares, one slot per parameter (_norm_index), zeros at
        # the window's start; _present: the parameters whose gradient the window applies; _stored: (parameter id, weak
        # reference, version) of the stored gradients the window's sums were taken from (world size N: the flat bucket's),
        # re-taken after step() and zero_grad(), so that a changed stored gradient marks a new window; _after_step: the
        # window's step() ran, its norms stay readable until the next window's first backward pass
        self._track = track_grad_norm_value(track_grad_norm)
        self._sums, self._present, self._stored, self._after_step = None, set(), None, False
        self._sumsq_ws = {}         # key -> workspace of a kernel that sums one tensor's squares (zeroed once)
        self._each_ws = None        # dd_grad_sumsq_each's workspace
        self._window_k = None       # factor of the window in progress, resolved at its first backward pass
        self._passes = {}           # id(wide param) -> backward passes that wrote its gradient in the window in progress
        self._acc_buf = {}          # world size 1: id(wide param) -> gradient buffer of passes 1 .. k-1 (allocated on first use)
        if len(self.param_groups) > 1 and dist.is_initialized() and dist.get_world_size(process_group) > 1:
            raise NotImplementedError("FusedAdam: the sharded form supports one parameter group")
        self.group = process_group
        self.world = dist.get_world_size(process_group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(process_group) if dist.is_initialized() else 0
        if self._clip_val and self.world > 1:
            raise NotImplementedError(_NO_SHARDED_CLIP)
        self._regions = {}          # id(param) -> region dict of a wide tensor
        self._flat = None           # region dict of the flat bucket
        self._symm = None
        self._overlap = bool(overlap_backward)
        self._defer_join = bool(defer_join)
        self._side = None           # stream of the updates launched from the backward pass
        self._written = set()       # ids of wide params whose gradient replica was written since the last step()
        self._launched = set()      # ... and whose update is already running on the side stream
        self._mom, self._mom_of = None, None   # symmetric buffer of this rank's moment shards, accessor for the peers'
        self._flat_mode = None      # world size N: how this window's flat-bucket norms were taken ("sharded" / "replicated")
        self._flat_replicated = False   # the flat bucket fell back to per-tensor replicated updates (partly frozen model)
        self._lib = _lib.load()     # raises when the CUDA library is missing: no fallback
        for g in self.param_groups:
            for p in g["params"]:
                self._check_param(p)
        self._fused = {}            # id(param) -> True once its step ran inside the backward pass (world size 1)
        self._norm_index = {id(p): i for i, p in enumerate(p for g in self.param_groups for p in g["params"])}
        self._slots = None          # world size N: this rank's fp64 shard sums, [wide regions | flat tensors] (symmetric)
        if self.world > 1:
            self._setup_sharding(shard_min_numel, multicast, broadcast_init)
        elif overlap_backward or fuse_into_backward:
            self._setup_fused_backward(shard_min_numel)

    # The two places where the device is touched outside `_launch_sharded`; tests/test_optim.py overrides them (and the
    # launch) to run the sharding logic itself under gloo on CPU tensors.
    def _check_param(self, p):
        if not (p.is_cuda and p.dtype == torch.float32 and p.is_contiguous()):
            raise RuntimeError("FusedAdam: parameters must be contiguous fp32 CUDA tensors")

    def _alloc_symmetric(self, numel, device, multicast):
        """One symmetric-memory buffer of `numel` floats per rank -> (buffer, handle with .barrier(channel=),
        per-rank device pointers, multicast address or 0)."""
        import torch.distributed._symmetric_memory as symm_mem
        buf = symm_mem.empty(numel, dtype=torch.float32, device=device)
        grp = self.group if self.group is not None else dist.group.WORLD
        hdl = symm_mem.rendezvous(buf, grp)
        # per NVLink direction and GPU the multicast form moves n(1 + 1/N) bytes (the switch also loops the own replica
        # back), peer loads / stores 2n(N-1)/N.  Alone, the multicast update is the shorter kernel from N = 6 on (2.0 vs
        # 3.0 ms at N = 8), but it runs BESIDE the conv backward pass, and multimem traffic slows those HBM-bound kernels far
        # more than peer loads do (N = 8, profiles/r2_step_timeline_n8_*.txt: input-gradient conv 1.36 vs 0.82 ms, c3
        # weight gradient 0.69 vs 0.28): 6.68 vs 6.46 ms per step at N = 8, 6.24 vs 5.66 at N = 2.  Peer loads by default.
        want_mc = False if multicast is None else bool(multicast)
        mc = int(hdl.multicast_ptr) if (want_mc and hdl.has_multicast_support) else 0
        if multicast is True and mc == 0:
            raise RuntimeError("FusedAdam: multicast requested but the symmetric buffer has no multicast mapping")
        return buf, hdl, [int(x) for x in hdl.buffer_ptrs], mc

    def _alloc_moments(self, numel, device):
        """Symmetric buffer for the moment shards -> (local tensor, fn(rank) -> that rank's tensor)."""
        import torch.distributed._symmetric_memory as symm_mem
        buf = symm_mem.empty(numel, dtype=torch.float32, device=device)
        grp = self.group if self.group is not None else dist.group.WORLD
        hdl = symm_mem.rendezvous(buf, grp)
        buf.zero_()
        return buf, (lambda rk: buf if rk == self.rank else hdl.get_buffer(rk, (numel,), torch.float32))

    @staticmethod
    def _alias(view):
        """A tensor over the same device memory as `view` but with a storage of its own, exactly as long as the tensor:
        torch.save of a parameter that is a plain view would serialise the whole [gradients | weights] buffer."""
        if view.device.type != "cuda":
            return view

        class _Mem:
            __cuda_array_interface__ = {"shape": tuple(view.shape), "typestr": "<f4", "data": (view.data_ptr(), False),
                                        "version": 3, "strides": None}

        return torch.as_tensor(_Mem(), device=view.device)

    # ------------------------------------------------------------------------------------------
    def _setup_sharding(self, shard_min_numel, multicast, broadcast_init):
        params = [p for g in self.param_groups for p in g["params"]]
        if broadcast_init:          # replicas must start identical (Lightning ddp broadcasts rank 0's weights)
            src = dist.get_global_rank(self.group, 0) if self.group is not None else 0
            for p in params:
                dist.broadcast(p.data, src=src, group=self.group)
        wide = [p for p in params if p.numel() >= shard_min_numel and p.numel() % 4 == 0]
        small = [p for p in params if not any(p is q for q in wide)]
        offs, flat_off = flat_layout([p.numel() for p in wide])
        small_offs, small_total = flat_layout([p.numel() for p in small])
        total = flat_off + small_total
        if total == 0:
            return
        dev = params[0].device
        buf, hdl, ptrs, mc = self._alloc_symmetric(2 * total, dev, multicast)      # [gradients | weights]
        buf.zero_()

        def adopt(p, off):
            n = p.numel()
            w = self._alias(buf[total + off: total + off + n].view_as(p))
            w.copy_(p.data)
            p.data = w                                   # the module now computes from the symmetric replica
            return buf[off: off + n].view_as(p)

        for p, off in zip(wide, offs):
            gview = adopt(p, off)
            p.grad = gview
            p._dd_grad_buffer = gview                    # ops.linear's weight-gradient kernel writes here ...
            p._dd_grad_begin = (lambda q: (lambda: self._begin_grad(q)))(p)          # (overwrite, or accumulate?)
            p._dd_grad_ready = (lambda q: (lambda: self._on_grad_written(q)))(p)     # ... and then calls this
            lo, hi = shard_bounds(p.numel(), self.world, self.rank)
            self._regions[id(p)] = dict(off=off, n=p.numel(), lo=lo, hi=hi, channel=1 + len(self._regions), key=p)
        if small:
            views = [adopt(p, flat_off + o) for p, o in zip(small, small_offs)]
            lo, hi = shard_bounds(small_total, self.world, self.rank)
            self._flat = dict(off=flat_off, n=small_total, lo=lo, hi=hi, channel=0, params=small, grad_views=views, key="flat",
                              offs=small_offs)
        # moment shards: [exp_avg | exp_avg_sq] per region, capacity = the longest shard (the last rank's), in a symmetric
        # buffer of their own so that state_dict() can read the peers' shards
        moff = 0
        for r in list(self._regions.values()) + ([self._flat] if self._flat is not None else []):
            lo_l, hi_l = shard_bounds(r["n"], self.world, self.world - 1)
            cap = -(-max(hi_l - lo_l, r["hi"] - r["lo"], 4) // _ALIGN) * _ALIGN
            r["moff"], r["mcap"] = moff, cap
            moff += 2 * cap
        # the norm slots (fp64) ride at the end of the same symmetric buffer: one per wide region, then one per flat tensor
        n_slots = len(self._regions) + len(small)
        moff += moff & 1
        self._mom, self._mom_of = self._alloc_moments(moff + 2 * n_slots, dev)
        self._slots = (moff, n_slots)
        self._norm_index = {id(p): i for i, p in enumerate([r["key"] for r in self._regions.values()] + small)}
        self._symm = dict(buf=buf, hdl=hdl, total=total, ptrs=ptrs, mc=mc)
        if self._overlap:
            self._side = torch.cuda.Stream(device=dev)
        if dev.type == "cuda":
            torch.cuda.synchronize()
        hdl.barrier()

    def _setup_fused_backward(self, min_numel):
        """World size 1, ``overlap_backward=True`` (``fuse_into_backward=True`` names the same form): the wide 2-D weights
        (the FC layers: > 99.9 % of the parameters) get their Adam step INSIDE the backward pass.  ops.linear's backward
        then runs one kernel per layer (dd_linear_bwd_adam) that streams each weight tile and its two moments through shared
        memory once: the input gradient is computed from the old weight, the weight gradient is consumed on chip where it is
        produced, and the updated weight and moments are written back -- 24 bytes per parameter instead of the 40 of the
        input-gradient, weight-gradient and Adam kernels, and no gradient buffers (1.3 GB less for RoadMapBCE).  Results are
        those of the unfused form.  step() then skips these weights.  With accumulate_grad_batches = 1 ops.linear falls back
        to a stored gradient whenever the fused kernel does not apply (batch > 32, CUDA-core path), and step() handles that;
        with k > 1 every backward pass of these weights comes here (_window_backward)."""
        for g in self.param_groups:
            for p in g["params"]:
                if p.dim() == 2 and p.numel() >= min_numel and p.is_cuda:
                    p._dd_fused_update = _BackwardHook(self, g, p)

    def _factor(self):
        """accumulate_grad_batches of the window in progress (a schedule is resolved at the window's first pass)."""
        if self._window_k is None:
            self._window_k = accumulation_factor(self.accumulate_grad_batches, self.current_epoch())
        return self._window_k

    def _refuse_pass(self, n, what):
        raise RuntimeError(f"FusedAdam: backward pass {n} without a step() in between reached {what}, but "
                           f"accumulate_grad_batches={self._window_k} (set it to accumulate more passes per step)")

    @torch.no_grad()
    def _window_backward(self, g, p, dy, x, w, dx, db, ws, ws_bytes, fusable, impl):
        """World size 1, accumulate_grad_batches = k > 1: one backward pass of a wide weight.  Passes 1 .. k-1 compute the
        input gradient and add the weight gradient into the weight's buffer (the first pass overwrites it); pass k runs
        dd_linear_bwd_adam_acc (the step folded in) where the fused kernel applies, else it adds into the buffer as well and
        step() steps from there."""
        key = id(p)
        k = self._factor()
        j = self._passes.get(key, 0)
        if j >= k or key in self._fused:
            self._refuse_pass(j + 1, "a weight whose window is complete")
        B, K = x.shape
        N = p.shape[0]
        buf = self._acc_buf.get(key)
        if buf is None:
            buf = self._acc_buf[key] = torch.empty_like(p)
        if j == 0:
            self._window_starts()
        if j + 1 == k and fusable:
            st = self._state(p, p.numel(), p.device)
            st["step"] += 1
            args = (dy.data_ptr(), x.data_ptr(), p.data_ptr(), st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr(),
                    buf.data_ptr(), dx.data_ptr() if dx is not None else None,
                    _lib.dtype_code(dx.dtype) if dx is not None else _lib.DD_F32, db.data_ptr() if db is not None else None,
                    ws.data_ptr(), ws_bytes, B, N, K, float(g["lr"]), float(g["betas"][0]), float(g["betas"][1]),
                    float(g["eps"]), float(g["weight_decay"]), st["step"])
            if self._track:
                call("dd_linear_bwd_adam_sumsq", *args, *self._sumsq_slot(p), stream_ptr())
            else:
                call("dd_linear_bwd_adam_acc", *args, stream_ptr())
            self._fused[key] = True
        else:
            if dx is not None:
                call("dd_linear_dgrad", dy.data_ptr(), w.data_ptr(), dx.data_ptr(), _lib.dtype_code(dx.dtype), ws.data_ptr(),
                     ws_bytes, B, N, K, impl, stream_ptr())
            call("dd_linear_wgrad_acc", dy.data_ptr(), x.data_ptr(), _lib.dtype_code(x.dtype), buf.data_ptr(),
                 db.data_ptr() if db is not None else None, B, N, K, impl, int(j > 0), stream_ptr())
        self._passes[key] = j + 1

    @torch.no_grad()
    def _fused_step(self, g, p, dy, x, dx, db, ws, ws_bytes):
        if id(p) in self._fused:
            raise RuntimeError("FusedAdam: two backward passes reached a weight whose Adam step is folded into its backward, "
                               "without a step() in between")
        self._window_starts()
        st = self._state(p, p.numel(), p.device)
        st["step"] += 1
        B, K = x.shape
        dxa = (dx.data_ptr() if dx is not None else None, _lib.dtype_code(dx.dtype) if dx is not None else _lib.DD_F32)
        args = (db.data_ptr() if db is not None else None, ws.data_ptr(), ws_bytes, B, p.shape[0], K, float(g["lr"]),
                float(g["betas"][0]), float(g["betas"][1]), float(g["eps"]), float(g["weight_decay"]), st["step"])
        head = (dy.data_ptr(), x.data_ptr(), p.data_ptr(), st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr())
        if self._track:
            call("dd_linear_bwd_adam_sumsq", *head, None, *dxa, *args, *self._sumsq_slot(p), stream_ptr())
        else:
            call("dd_linear_bwd_adam", *head, *dxa, *args, stream_ptr())
        self._fused[id(p)] = True

    @property
    def gradient_clip_val(self) -> float:
        """max_norm of the clip_grad_norm_ every step applies (0 = off).  It decides whether a wide weight's step may run
        inside the backward pass, so it changes between steps only: not after a backward pass of a window whose step()
        has not run yet."""
        return self._clip_val

    @gradient_clip_val.setter
    def gradient_clip_val(self, c):
        c = gradient_clip_value(c)
        if c and self.world > 1:
            raise NotImplementedError(_NO_SHARDED_CLIP)
        if c != self._clip_val and (self._passes or self._fused or self._written):
            raise RuntimeError("FusedAdam: gradient_clip_val cannot change after a backward pass of a window whose step() "
                               "has not run; change it between steps")
        self._clip_val = c

    @property
    def track_grad_norm(self):
        """2 when grad_norms() tracks the 2-norm, else -1 (off).  It decides which kernels the backward pass launches, so it
        changes between steps only."""
        return 2 if self._track else -1

    @track_grad_norm.setter
    def track_grad_norm(self, t):
        on = track_grad_norm_value(t)
        if on != self._track and (self._passes or self._fused or self._written):
            raise RuntimeError("FusedAdam: track_grad_norm cannot change after a backward pass of a window whose step() "
                               "has not run; change it between steps")
        self._track = on

    @property
    def uses_multicast(self) -> bool:
        return bool(self._symm and self._symm["mc"])

    # ------------------------------------------------------------------------------------------
    def zero_grad(self, set_to_none: bool = True):
        # an unfinished accumulation window is discarded (its next pass overwrites the gradient buffer again); a finished
        # one -- its update already launched or folded into the backward pass -- is left for step()
        k = self._window_k
        for key, n in list(self._passes.items()):
            if n < k and key not in self._fused:
                del self._passes[key]
                self._written.discard(key)
        if not self._passes and not self._written and not self._fused:
            self._window_k = None
        for g in self.param_groups:
            for p in g["params"]:
                if id(p) in self._regions:       # persistent view of the symmetric buffer, overwritten by every backward
                    continue
                if p.grad is None:
                    continue
                if set_to_none:
                    p.grad = None
                else:
                    p.grad.detach_()
                    p.grad.zero_()
        if self._after_step:                     # clearing the gradients starts no window: only a backward pass does
            self._stored = self._fingerprint(self._stored_todo())

    def _state(self, key, numel, device):
        st = self.state[key]
        if not st:
            st["step"] = 0
            st["exp_avg"] = torch.zeros(numel, dtype=torch.float32, device=device)
            st["exp_avg_sq"] = torch.zeros(numel, dtype=torch.float32, device=device)
        return st

    def _shard_state(self, r):
        """State of a sharded region: views of this rank's piece of the symmetric moments buffer."""
        st = self.state[r["key"]]
        if not st:
            n = r["hi"] - r["lo"]
            st["step"] = 0
            st["exp_avg"] = self._mom[r["moff"]: r["moff"] + n]
            st["exp_avg_sq"] = self._mom[r["moff"] + r["mcap"]: r["moff"] + r["mcap"] + n]
        return st

    def _hyper(self):
        g = self.param_groups[0]
        return (float(g["lr"]), float(g["betas"][0]), float(g["betas"][1]), float(g["eps"]), float(g["weight_decay"]))

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        self._window_k = None
        if self.world == 1:
            todo = self._local_todo()
            if self._track:
                if self._after_step:                      # no backward pass reached a wide weight since the last step
                    self._window_starts()
                self._stored_sums(todo)
            if self.gradient_clip_val:
                todo = [(g, p, _f32(grad)) for g, p, grad in todo]
                coef = self._clip([grad for _, _, grad in todo])
                for g, p, grad in todo:
                    self._launch_local(g, p, grad, coef)
            else:
                for g, p, grad in todo:
                    self._launch_local(g, p, grad)
            self._fused.clear()
            self._passes.clear()
            self._stepped()
            return loss
        if self._symm is None:
            return loss
        if self._track and self._after_step:             # no backward pass reached a wide weight since the last step
            self._window_starts()
        hdl = self._symm["hdl"]
        todo = [r for key, r in self._regions.items() if key in self._written and key not in self._launched]
        fl, restage = self._flat, False
        if fl is not None:
            have = [p.grad is not None for p in fl["params"]]
            if any(have) and (self._flat_replicated or not all(have)):
                # A partly frozen bucket (e.g. RoadMapBCE before unfreeze_epoch_no, roadmap_bce_v2.py:127-129):
                # torch.optim.Adam skips tensors without a gradient and keeps a step count per tensor, which one sharded
                # bucket cannot express.  These tensors are 0.1 % of the bytes: average each present gradient with an
                # all-reduce and update every replica locally, per tensor -- and stay in this form from then on, so the
                # per-tensor moments remain the truth.
                if self.state.get("flat"):
                    raise NotImplementedError("FusedAdam (world > 1): the flat bucket was already stepped in its sharded form; "
                                              "freeze parameters before the first step, not after")
                self._flat_replicated = True
                # grad_norms() took its sums from an all-reduced copy; from the averaged p.grad if they changed since
                renorm = self._track and self._flat_stale()
                nccl = dist.get_backend(self.group) == "nccl"
                g = self.param_groups[0]
                for p in fl["params"]:
                    if p.grad is None:
                        continue
                    dist.all_reduce(p.grad, op=dist.ReduceOp.AVG if nccl else dist.ReduceOp.SUM, group=self.group)
                    if not nccl:
                        p.grad.div_(self.world)
                    self._launch_local(g, p, p.grad)
                if renorm:
                    self._flat_norms_replicated([p.grad for p in fl["params"] if p.grad is not None])
            elif all(have):
                restage = self._flat_mode != "sharded" or self._flat_stale()
                if restage:                            # else grad_norms() staged these very gradients
                    torch._foreach_copy_(fl["grad_views"], [p.grad for p in fl["params"]])
                todo.append(fl)
        if todo:
            hdl.barrier()                                  # every rank has written its gradient replicas
            if self._track and fl is not None and todo[-1] is fl and restage:
                self._flat_norms_sharded()                 # read before the closing barrier: no replica changes under it
            for r in todo:
                self._launch_region(r, ctas_per_sm=8)
            hdl.barrier()                                  # every replica holds the new weights
        if self._launched:
            # The updates launched from the backward pass run on the side stream and end with a cross-rank barrier (new
            # weights landed in every replica, every rank done reading the gradient replicas).  Their tail (the NVLink
            # exchange of the last wide tensor) need not finish before step() returns -- only before the next READ of that
            # weight: each adopted parameter carries an event that ops.linear waits for in the next forward pass, so the tail
            # overlaps with the next step's conv forward instead of being exposed (N = 8: ~1 ms per step).  synchronize()
            # joins explicitly (checkpointing, evaluation code that reads the parameters directly).
            if self._defer_join:
                ev = torch.cuda.Event()
                ev.record(self._side)
                for key in self._launched:
                    self._regions[key]["key"]._dd_ready_event = ev
                self._pending = ev
            else:
                torch.cuda.current_stream().wait_stream(self._side)
        self._launched.clear()
        self._written.clear()
        self._passes.clear()
        self._stepped()
        return loss

    def synchronize(self):
        """Make the current stream wait for weight updates still running on the side stream (overlap_backward)."""
        ev = getattr(self, "_pending", None)
        if ev is not None:
            torch.cuda.current_stream().wait_event(ev)
            self._pending = None

    # ------------------------------------------------------------------------------------------
    # checkpointing: torch.optim.Adam's layout in and out
    # ------------------------------------------------------------------------------------------
    def _full_moments(self, r):
        """(exp_avg, exp_avg_sq) of a sharded region at full length, assembled from every rank's shard."""
        dev = self._mom.device
        if dev.type == "cuda":
            torch.cuda.synchronize(dev)      # this rank's step() ended with a cross-rank barrier: every shard is up to date
        m, v = torch.empty(r["n"], dtype=torch.float32, device=dev), torch.empty(r["n"], dtype=torch.float32, device=dev)
        for rk in range(self.world):
            lo, hi = shard_bounds(r["n"], self.world, rk)
            peer = self._mom_of(rk)
            m[lo:hi].copy_(peer[r["moff"]: r["moff"] + hi - lo])
            v[lo:hi].copy_(peer[r["moff"] + r["mcap"]: r["moff"] + r["mcap"] + hi - lo])
        return m, v

    def state_dict(self):
        self.synchronize()
        index, groups = {}, []
        for g in self.param_groups:
            pg = {k: v for k, v in g.items() if k != "params"}
            pg["params"] = []
            for p in g["params"]:
                index[id(p)] = len(index)
                pg["params"].append(index[id(p)])
            groups.append(pg)
        state = {}

        def put(p, step, m, v):
            state[index[id(p)]] = {"step": torch.tensor(float(step), dtype=torch.float32),
                                   "exp_avg": m.detach().clone().view_as(p), "exp_avg_sq": v.detach().clone().view_as(p)}

        for g in self.param_groups:
            for p in g["params"]:
                st = self.state.get(p)
                if st and id(p) not in self._regions:        # world 1, or the per-tensor (replicated) form
                    put(p, st["step"], st["exp_avg"], st["exp_avg_sq"])
        for key, r in self._regions.items():
            st = self.state.get(r["key"])
            if st and not isinstance(r["key"], str):
                m, v = self._full_moments(r)
                put(r["key"], st["step"], m, v)
        fl = self._flat
        if fl is not None and self.state.get("flat"):
            m, v = self._full_moments(fl)
            for p, o in zip(fl["params"], fl["offs"]):
                put(p, self.state["flat"]["step"], m[o: o + p.numel()], v[o: o + p.numel()])
        return {"state": state, "param_groups": groups}

    def load_state_dict(self, state_dict):
        params = [p for g in self.param_groups for p in g["params"]]
        saved_groups = state_dict["param_groups"]
        ids = [i for g in saved_groups for i in g["params"]]
        if len(ids) != len(params):
            raise ValueError("FusedAdam.load_state_dict: the checkpoint has a different number of parameters")
        for g, sg in zip(self.param_groups, saved_groups):
            for k, v in sg.items():
                if k != "params" and k in g:
                    g[k] = v
        by_param = {id(p): state_dict["state"].get(i, state_dict["state"].get(str(i))) for p, i in zip(params, ids)}

        def unpack(p):
            st = by_param.get(id(p))
            if not st:
                return None
            step = st["step"]
            step = int(round(float(step.item() if torch.is_tensor(step) else step)))
            dev = p.device
            m = st["exp_avg"].detach().to(device=dev, dtype=torch.float32).reshape(-1)
            v = st["exp_avg_sq"].detach().to(device=dev, dtype=torch.float32).reshape(-1)
            if m.numel() != p.numel():
                raise ValueError("FusedAdam.load_state_dict: moment shape does not match the parameter")
            return step, m, v

        self.state.clear()
        for p in params:
            if id(p) in self._regions:
                got = unpack(p)
                if got:
                    r = self._regions[id(p)]
                    st = self._shard_state(r)
                    st["step"] = got[0]
                    st["exp_avg"].copy_(got[1][r["lo"]: r["hi"]])
                    st["exp_avg_sq"].copy_(got[2][r["lo"]: r["hi"]])
        fl = self._flat
        flat_ids = {id(p) for p in fl["params"]} if fl is not None else set()
        if fl is not None:
            got = [unpack(p) for p in fl["params"]]
            steps = {g[0] for g in got if g}
            if all(got) and len(steps) == 1:                 # one step count: the sharded form can carry it
                dev = self._mom.device
                m, v = torch.zeros(fl["n"], device=dev), torch.zeros(fl["n"], device=dev)
                for p, o, g in zip(fl["params"], fl["offs"], got):
                    m[o: o + p.numel()].copy_(g[1])
                    v[o: o + p.numel()].copy_(g[2])
                st = self._shard_state(fl)
                st["step"] = steps.pop()
                st["exp_avg"].copy_(m[fl["lo"]: fl["hi"]])
                st["exp_avg_sq"].copy_(v[fl["lo"]: fl["hi"]])
                self._flat_replicated = False
            elif any(got):                                   # per-tensor step counts (partly frozen history): replicated form
                self._flat_replicated = True
                for p, g in zip(fl["params"], got):
                    if g:
                        self.state[p] = {"step": g[0], "exp_avg": g[1].clone(), "exp_avg_sq": g[2].clone()}
        for p in params:
            if id(p) in self._regions or id(p) in flat_ids:
                continue
            got = unpack(p)
            if got:
                self.state[p] = {"step": got[0], "exp_avg": got[1].clone(), "exp_avg_sq": got[2].clone()}

    def _clip(self, grads):
        """clip_grad_norm_'s total norm and coefficient over `grads` (contiguous fp32), on the device: one dd_grad_sumsq
        call.  Sets last_grad_norm; returns the coefficient (a 1-element device tensor)."""
        dev = self.param_groups[0]["params"][0].device
        if self._clip_ws is None:
            self._clip_ws = torch.zeros(int(self._lib.dd_grad_sumsq_workspace_bytes()), dtype=torch.uint8, device=dev)
        out = torch.empty(4, dtype=torch.float32, device=dev)       # norm, coefficient, fp64 sum of squares
        n = len(grads)
        call("dd_grad_sumsq", (ctypes.c_void_p * n)(*[t.data_ptr() for t in grads]),
             (ctypes.c_longlong * n)(*[t.numel() for t in grads]), n, self.gradient_clip_val, out.data_ptr(),
             self._clip_ws.data_ptr(), self._clip_ws.numel(), stream_ptr())
        self.last_grad_norm = out[0]
        return out[1:]

    def _launch_local(self, g, p, grad, coef=None):
        """One dd_adam_step launch: the whole tensor, this replica only (dd_adam_step_clipped with a clip coefficient)."""
        grad = _f32(grad)
        st = self._state(p, p.numel(), p.device)
        st["step"] += 1
        args = (p.data_ptr(), grad.data_ptr(), st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr(), p.numel(),
                float(g["lr"]), float(g["betas"][0]), float(g["betas"][1]), float(g["eps"]), float(g["weight_decay"]),
                st["step"], 1.0)
        if coef is None:
            call("dd_adam_step", *args, stream_ptr())
        else:
            call("dd_adam_step_clipped", *args, coef.data_ptr(), stream_ptr())

    def _launch_region(self, r, ctas_per_sm):
        """The sharded update of a region; with tracking, a wide region's also writes this rank's shard sum of squares into
        the region's norm slot (the flat bucket's per-tensor sums come from _flat_norms_*)."""
        if self._track and r is not self._flat:
            self._present.add(id(r["key"]))
            self._launch_sharded(r, ctas_per_sm=ctas_per_sm, norm=True)
        else:
            self._launch_sharded(r, ctas_per_sm=ctas_per_sm)

    def _launch_sharded(self, r, ctas_per_sm, norm=False):
        sy, W = self._symm, self.world
        lo, hi, total = r["lo"], r["hi"], sy["total"]
        st = self._shard_state(r)
        st["step"] += 1
        gptrs = (ctypes.c_void_p * W)(*[b + 4 * r["off"] for b in sy["ptrs"]])
        wptrs = (ctypes.c_void_p * W)(*[b + 4 * (total + r["off"]) for b in sy["ptrs"]])
        mcg = ctypes.c_void_p(sy["mc"] + 4 * r["off"]) if sy["mc"] else None
        mcw = ctypes.c_void_p(sy["mc"] + 4 * (total + r["off"])) if sy["mc"] else None
        lr, b1, b2, eps, wd = self._hyper()
        args = (gptrs, wptrs, mcg, mcw, W, self.rank, st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr(), lo, hi - lo, lr, b1,
                b2, eps, wd, st["step"], 1.0 / W, int(ctas_per_sm))
        if norm:
            ws = self._sumsq_workspace(r["channel"])
            call("dd_adam_step_sharded_sumsq", *args, self._slot_ptr(self._norm_index[id(r["key"])]), ws.data_ptr(), ws.numel(),
                 stream_ptr())
        else:
            call("dd_adam_step_sharded", *args, stream_ptr())

    # ------------------------------------------------------------------------------------------
    # gradient norms (track_grad_norm)
    # ------------------------------------------------------------------------------------------
    def grad_norms(self):
        """{param: L2 norm of the gradient the window's step applies, a 0-dim fp32 device tensor} for every parameter with a
        gradient in the window, plus ``"total"``, the norm of all of them together.  The gradient is the window's (summed
        over accumulate_grad_batches passes), the rank mean at world size N, before any clipping.  No host sync.  Valid
        from the window's last backward pass (before or after step()) until the next window's first backward pass; outside
        that range it raises.  At world size N every rank must call it (it may exchange the flat bucket's gradients), and
        every rank gets the same bits; with overlap_backward=False the wide weights update inside step(), so their norms
        exist only after it."""
        if not self._track:
            raise RuntimeError("FusedAdam.grad_norms: track_grad_norm is off (set track_grad_norm=2)")
        if self.world == 1:
            if self._after_step and self._changed(self._stored, self._local_todo()):
                # a backward pass wrote stored gradients since step() (zero_grad() alone does not count)
                if any(hasattr(p, "_dd_fused_update") for g in self.param_groups for p in g["params"]):
                    raise RuntimeError("FusedAdam.grad_norms: the next window's backward pass has begun; its norms are "
                                       "valid once the window's last backward pass has run")
                self._window_starts()                    # stored gradients only: a new window's gradients
            if not self._after_step:
                self._check_window_complete()
                self._stored_sums(self._local_todo())
        else:
            self._dist_sums()
        return self._result()

    def _window_starts(self):
        """The first backward pass of a window after a step(): the previous window's norms are gone."""
        if self._after_step:
            self._sums, self._present, self._stored, self._after_step = None, set(), None, False
            self._flat_mode = None

    def _window_sums(self):
        if self._sums is None:
            dev = self.param_groups[0]["params"][0].device
            self._sums = torch.zeros(len(self._norm_index), dtype=torch.float64, device=dev)
        return self._sums

    def _sumsq_workspace(self, key):
        ws = self._sumsq_ws.get(key)
        if ws is None:
            dev = self.param_groups[0]["params"][0].device
            ws = self._sumsq_ws[key] = torch.zeros(int(self._lib.dd_grad_sumsq_workspace_bytes()), dtype=torch.uint8, device=dev)
        return ws

    def _sumsq_slot(self, p):
        """(sum pointer, workspace pointer, workspace bytes) for the fused kernel stepping p at world size 1."""
        self._present.add(id(p))
        ws = self._sumsq_workspace(id(p))
        return self._window_sums()[self._norm_index[id(p)]].data_ptr(), ws.data_ptr(), ws.numel()

    def _slot_ptr(self, i):
        """Device address of this rank's norm slot i (world size N)."""
        return self._mom.data_ptr() + 4 * self._slots[0] + 8 * i

    def _local_todo(self):
        """World size 1: (group, param, gradient) of every tensor step() applies from a stored gradient."""
        todo = []
        for g in self.param_groups:
            for p in g["params"]:
                if id(p) in self._fused:              # stepped inside the backward pass
                    continue
                if id(p) in self._passes:             # accumulation buffer: a window without the fused last pass
                    todo.append((g, p, self._acc_buf[id(p)]))
                elif p.grad is not None:
                    todo.append((g, p, p.grad))
        return todo

    @staticmethod
    def _fingerprint(todo):
        return [(id(p), weakref.ref(grad), grad._version) for _, p, grad in todo]

    @staticmethod
    def _changed(fp, todo):
        """`todo` (group, param, gradient) is not the set of tensors, at the versions, that fingerprint `fp` recorded."""
        return fp is None or len(todo) != len(fp) or any(
            key != id(p) or ref() is not grad or grad._version != v for (_, p, grad), (key, ref, v) in zip(todo, fp))

    def _stored_todo(self):
        """The stored gradients whose sums grad_norms() takes itself: world size 1 what step() applies from a stored
        gradient, world size N the flat bucket's."""
        if self.world == 1:
            return self._local_todo()
        return [(None, p, p.grad) for p in (self._flat["params"] if self._flat is not None else []) if p.grad is not None]

    def _flat_stale(self):
        return self._flat_mode is None or self._changed(self._stored, self._stored_todo())

    def _stepped(self):
        """End of step(): the window's norms stay readable, against the stored gradients as step() leaves them."""
        self._after_step = self._track
        if self._track:
            self._stored = self._fingerprint(self._stored_todo())

    def _stored_sums(self, todo):
        """World size 1: the sums of squares of the stored gradients `todo` (once per window; again if they changed)."""
        if not self._changed(self._stored, todo):
            return
        sums = self._window_sums()
        self._sumsq_each([_f32(grad) for _, _, grad in todo], [sums[self._norm_index[id(p)]] for _, p, _ in todo])
        self._present.update(id(p) for _, p, _ in todo)
        self._stored = self._fingerprint(todo)

    def _check_window_complete(self):
        k = self._window_k
        for key, n in self._passes.items():
            if key not in self._fused and key not in self._launched and k is not None and n < k:
                raise RuntimeError(f"FusedAdam.grad_norms: the window has run {n} of its {k} backward passes "
                                   "(accumulate_grad_batches); its norms exist after its last backward pass")

    def _mean_copies(self):
        """World size N, replicated flat form, before step(): the rank mean of each present gradient, by the all-reduce
        step() runs, on a copy -- p.grad stays this rank's, for whatever the training loop does before step()."""
        nccl = dist.get_backend(self.group) == "nccl"
        out = []
        for p in self._flat["params"]:
            if p.grad is None:
                continue
            t = p.grad.clone()
            dist.all_reduce(t, op=dist.ReduceOp.AVG if nccl else dist.ReduceOp.SUM, group=self.group)
            out.append(t if nccl else t.div_(self.world))
        return out

    def _flat_norms_replicated(self, means):
        """Per-tensor sums of the rank means `means` of the flat bucket's present gradients (the same bits on every
        rank)."""
        fl, sums = self._flat, self._window_sums()
        ps = [p for p in fl["params"] if p.grad is not None]
        self._sumsq_each(means, [sums[self._norm_index[id(p)]] for p in ps])
        self._present.update(id(p) for p in ps)
        self._flat_mode = "replicated"
        self._stored = self._fingerprint(self._stored_todo())

    def _flat_norms_sharded(self):
        """This rank's part of the flat bucket's per-tensor sums: its shard of each tensor, the rank mean as the sharded
        update consumes it, into the tensor's norm slot.  Between a barrier after every replica is written and one before
        any is written again."""
        fl = self._flat
        offs, numels, outs = [], [], []
        for p, o in zip(fl["params"], fl["offs"]):
            a, b = max(o, fl["lo"]), min(o + p.numel(), fl["hi"])
            offs.append(fl["off"] + (a if b > a else fl["lo"]))
            numels.append(max(b - a, 0))
            outs.append(self._norm_index[id(p)])
        self._sumsq_each_replicas(offs, numels, outs)
        self._present.update(id(p) for p in fl["params"])
        self._flat_mode = "sharded"
        self._stored = self._fingerprint(self._stored_todo())

    def _dist_sums(self):
        """World size N: the window's sums -- each wide region's and (sharded form) each flat tensor's from the N ranks'
        slots, added in rank order, so every rank holds the same bits."""
        if self._side is not None:
            torch.cuda.current_stream().wait_stream(self._side)     # its launches end with the cross-rank barrier
        if self._after_step and self._changed(self._stored, self._stored_todo()):
            self._window_starts()        # a backward pass wrote the flat gradients since step(): no wide weight started it
        if not self._after_step:
            for key in self._written:
                if key not in self._launched:
                    if not self._overlap:
                        raise RuntimeError("FusedAdam.grad_norms: with overlap_backward=False the data-parallel form updates "
                                           "the wide weights inside step(), so their norms exist only after step()")
                    self._check_window_complete()
            fl = self._flat
            if fl is not None and self._flat_stale():
                have = [p.grad is not None for p in fl["params"]]
                if any(have) and (self._flat_replicated or not all(have)):
                    self._flat_norms_replicated(self._mean_copies())
                elif all(have):
                    # staged into the replica here; step() copies again only if p.grad changed since (e.g. a clip)
                    torch._foreach_copy_(fl["grad_views"], [p.grad for p in fl["params"]])
                    hdl = self._symm["hdl"]
                    hdl.barrier()                              # every rank has written its flat gradient replica
                    self._flat_norms_sharded()
                    hdl.barrier()                              # every rank's flat slots are written
        base, n = self._slots
        acc = None
        for rk in range(self.world):                           # rank order: the same bits on every rank
            t = self._mom_of(rk)[base: base + 2 * n].view(torch.float64)
            acc = t.clone() if acc is None else acc.add_(t)
        sums = self._window_sums()
        regions = list(self._regions.values())
        R = len(regions)
        sums[:R].copy_(acc[:R])
        for i, r in enumerate(regions):
            if id(r["key"]) not in self._present:
                sums[i].zero_()
        if self._flat_mode == "sharded":
            sums[R:].copy_(acc[R:])

    def _result(self):
        if not self._present:
            raise RuntimeError("FusedAdam.grad_norms: no gradient in this window yet; its norms exist after its last "
                               "backward pass")
        sums = self._sums
        norms = sums.sqrt().float()
        out = {p: norms[self._norm_index[id(p)]] for g in self.param_groups for p in g["params"] if id(p) in self._present}
        out["total"] = sums.sum().sqrt().float()
        return out

    # the device calls of the stored-gradient sums (tests/test_grad_norm_cpu.py emulates them)
    def _sumsq_each(self, grads, outs):
        if not grads:
            return
        dev = grads[0].device
        if self._each_ws is None:
            self._each_ws = torch.zeros(int(self._lib.dd_grad_sumsq_each_workspace_bytes()), dtype=torch.uint8, device=dev)
        n = len(grads)
        call("dd_grad_sumsq_each", (ctypes.c_void_p * n)(*[t.data_ptr() for t in grads]),
             (ctypes.c_longlong * n)(*[t.numel() for t in grads]), (ctypes.c_void_p * n)(*[o.data_ptr() for o in outs]), n,
             self._each_ws.data_ptr(), self._each_ws.numel(), stream_ptr())

    def _sumsq_each_replicas(self, offs, numels, slots):
        """Per-tensor sums of the flat bucket's rank mean over this rank's shard, into this rank's norm slots `slots`."""
        sy, n = self._symm, len(offs)
        outs = [self._slot_ptr(i) for i in slots]
        if self._each_ws is None:
            self._each_ws = torch.zeros(int(self._lib.dd_grad_sumsq_each_workspace_bytes()), dtype=torch.uint8,
                                        device=self._mom.device)
        call("dd_grad_sumsq_each_replicas", (ctypes.c_void_p * self.world)(*sy["ptrs"]), self.world, self.rank,
             1.0 / self.world, (ctypes.c_longlong * n)(*offs), (ctypes.c_longlong * n)(*numels), (ctypes.c_void_p * n)(*outs),
             n, self._each_ws.data_ptr(), self._each_ws.numel(), stream_ptr())

    def _begin_grad(self, p):
        """Called by ops.linear's backward before it writes p's gradient replica: 0 = overwrite (first pass of a window),
        1 = add to it (passes 2 .. k, dd_linear_wgrad_acc)."""
        n = self._passes.get(id(p), 0)
        if n >= self._factor():
            self._refuse_pass(n + 1, "a sharded parameter")
        if n == 0:
            self._window_starts()
        return int(n > 0)

    @torch.no_grad()
    def _on_grad_written(self, p):
        """Called by ops.linear's backward right after p's gradient replica is written.  overlap_backward: on the last
        pass of an accumulation window (every pass when accumulate_grad_batches = 1) the reduce + Adam + all-gather kernel
        is launched here, on a side stream, one 256-thread CTA per SM beside the persistent conv kernels of the rest of the
        backward pass; step() joins the side stream.  (The weights then change before step() is called: for training
        loops that step after every window, like the reference's.)  Earlier passes of a window stay on this rank."""
        key = id(p)
        k = self._factor()
        n = self._passes.get(key, 0) + 1
        if n > k:
            raise RuntimeError("FusedAdam: two backward passes wrote the gradient of a sharded parameter without a "
                               f"step() in between (accumulate_grad_batches={k}: a window of {k} passes per step)")
        self._passes[key] = n
        self._written.add(key)
        if not self._overlap or n < k:
            return
        r = self._regions[key]
        hdl = self._symm["hdl"]
        self._side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self._side):
            hdl.barrier(channel=r["channel"])
            self._launch_region(r, ctas_per_sm=1)
            hdl.barrier(channel=r["channel"])
        self._launched.add(key)


def follow_norm_tracking(hparams) -> int:
    """FusedAdam's track_grad_norm from the Namespace's (Lightning's flag; off when absent).  A norm FusedAdam cannot track
    is left to Lightning, with a warning."""
    t = getattr(hparams, "track_grad_norm", None) if hparams is not None else None
    try:
        return 2 if track_grad_norm_value(t) else -1
    except ValueError:
        warnings.warn(f"make_adam: FusedAdam cannot track the {t!r}-norm of the gradients (only the 2-norm); "
                      "track_grad_norm is left to Lightning, whose numbers miss the wide weights (their step runs inside "
                      "a kernel and they keep no .grad) and, under torch.distributed, are this rank's own gradients")
        return -1


def attach_optimizer(module, opt):
    """Record `opt` as the optimizer of `module` (its grad_norm() reads FusedAdam.grad_norms() from it), and let a
    checkpoint (module.state_dict()) see the weights of updates still in flight on the side stream."""
    module._dd_optimizer = opt
    if isinstance(opt, FusedAdam):
        module.register_state_dict_pre_hook(lambda *a, **k: opt.synchronize())


def _f32(grad):
    return grad if grad.is_contiguous() and grad.dtype == torch.float32 else grad.contiguous().float()


def follow_accumulation(opt, module):
    """Give FusedAdam the module's ``hparams.accumulate_grad_batches`` (1 when absent) and its ``current_epoch`` for an
    ``{epoch: factor}`` schedule."""
    hp = getattr(module, "hparams", None)
    acc = getattr(hp, "accumulate_grad_batches", None) if hp is not None else None
    accumulation_factor(1 if acc is None else acc)
    opt.accumulate_grad_batches = 1 if acc is None else acc
    opt.current_epoch = lambda: int(getattr(module, "current_epoch", 0) or 0)


def follow_clipping(hparams, distributed: bool) -> float:
    """FusedAdam's gradient_clip_val from the Namespace's (Lightning's flag; 0 when absent).  Under torch.distributed
    FusedAdam does not clip yet: the flag is then left to the Trainer, as it was before FusedAdam could clip, with a
    warning."""
    clip = gradient_clip_value(getattr(hparams, "gradient_clip_val", None))
    if clip and distributed:
        warnings.warn("make_adam: FusedAdam does not clip gradients under torch.distributed; gradient_clip_val is left to "
                      "the Trainer, whose clip misses the wide weights (they step inside the backward pass)")
        return 0.0
    return clip


class _BackwardHook:
    """``weight._dd_fused_update`` at world size 1: ops.linear's backward hands FusedAdam the weight's backward pass when
    ``takes(fusable)`` -- the fused backward + Adam kernel applies (``fusable``), or an accumulation window is open.  Under
    gradient clipping the step cannot run inside the backward pass (the norm needs every gradient first): the pass is never
    fusable then."""

    def __init__(self, opt, group, p):
        self.opt, self.group, self.p = opt, group, p

    def takes(self, fusable: bool) -> bool:
        return (fusable and not self.opt.gradient_clip_val) or self.opt._factor() > 1

    def __call__(self, dy, x, w, dx, db, ws, ws_bytes, fusable, impl):
        fusable = fusable and not self.opt.gradient_clip_val
        if self.opt._factor() == 1:
            self.opt._fused_step(self.group, self.p, dy, x, dx, db, ws, ws_bytes)
        else:
            self.opt._window_backward(self.group, self.p, dy, x, w, dx, db, ws, ws_bytes, fusable, impl)


def make_adam(module, lr):
    """What the task modules' ``configure_optimizers`` return for ``torch.optim.Adam(self.parameters(), lr)``
    (roadmap_bce_v2.py:155, autoencoder.py:120, spatial_w_rm.py:189).  hparams.optimizer = "fused" (the default when the
    model sits on a CUDA device): ``FusedAdam`` -- the dd_adam_step kernels, and under torch.distributed the sharded
    reduce + Adam + all-gather exchange, launched from the backward pass; "torch": the reference's optimizer object.
    ``hparams.accumulate_grad_batches`` (what Lightning's ``Trainer.add_argparse_args`` puts on the Namespace; an int or an
    ``{epoch: factor}`` dict, read against ``module.current_epoch`` at the first backward pass of each window) becomes
    FusedAdam's window of backward passes per step; ``hparams.gradient_clip_val`` (also the Trainer's flag) its clipping at
    world size 1.  Under torch.distributed FusedAdam does not clip yet: there the flag is left to the Trainer, as before
    FusedAdam could clip, with a warning.  ``hparams.track_grad_norm`` = 2 (the Trainer's flag too) turns on FusedAdam's
    gradient norms, which the module's grad_norm() returns; another norm is left to Lightning, with a warning."""
    hp = getattr(module, "hparams", None)
    kind = getattr(hp, "optimizer", "fused") if hp is not None else "fused"
    params = [p for p in module.parameters()]
    on_cuda = bool(params) and all(p.is_cuda for p in params)
    if kind == "fused" and on_cuda:
        distributed = dist.is_initialized() and dist.get_world_size() > 1
        opt = FusedAdam(params, lr=lr, overlap_backward=distributed, gradient_clip_val=follow_clipping(hp, distributed),
                        track_grad_norm=follow_norm_tracking(hp))
        follow_accumulation(opt, module)
        attach_optimizer(module, opt)
        return opt
    opt = torch.optim.Adam(params, lr=lr)
    attach_optimizer(module, opt)
    return opt
