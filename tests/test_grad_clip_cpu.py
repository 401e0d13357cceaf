"""Gradient clipping in optim.FusedAdam, host logic on CPU: the validation of gradient_clip_val, which gradients step()
hands dd_grad_sumsq and in what order relative to the Adam launches (device calls emulated), the backward-pass hook giving
up the fused update under clipping, changes of the flag between steps only, make_adam's reading of it, and the refusal of
clipping under torch.distributed."""
import math
import os
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cpu_adam_class():
    from driving_dirty_b200.optim import FusedAdam

    class CpuAdam(FusedAdam):
        """World size 1 on CPU tensors: dd_grad_sumsq and the Adam launches are recorded, not run."""

        def _check_param(self, p):
            assert p.dtype == torch.float32 and p.is_contiguous()

        def _clip(self, grads):
            self.log.append(("clip", [t.data_ptr() for t in grads]))
            total = math.sqrt(sum(float((t.double() ** 2).sum()) for t in grads))
            self.last_grad_norm = torch.tensor(total, dtype=torch.float32)
            return torch.tensor([min(self.gradient_clip_val / (total + 1e-6), 1.0)])

        def _launch_local(self, g, p, grad, coef=None):
            self.log.append(("adam", p.data_ptr(), grad.data_ptr(), None if coef is None else float(coef)))

    return CpuAdam


def test_gradient_clip_value():
    from driving_dirty_b200.optim import gradient_clip_value
    assert gradient_clip_value(None) == 0.0 and gradient_clip_value(0) == 0.0 and gradient_clip_value(0.5) == 0.5
    assert gradient_clip_value(2) == 2.0
    for bad in (-1.0, -1e-9, float("inf"), float("-inf"), float("nan"), True, "1"):
        with pytest.raises(ValueError, match="gradient_clip_val"):
            gradient_clip_value(bad)


def test_constructor_validates():
    CpuAdam = _cpu_adam_class()
    p = torch.nn.Parameter(torch.zeros(8))
    assert CpuAdam([p]).gradient_clip_val == 0.0
    assert CpuAdam([p], gradient_clip_val=None).gradient_clip_val == 0.0
    assert CpuAdam([p], gradient_clip_val=1).gradient_clip_val == 1.0
    for bad in (-1.0, float("nan"), float("inf")):
        with pytest.raises(ValueError):
            CpuAdam([p], gradient_clip_val=bad)


def test_clip_value_changes_between_steps_only():
    """The flag decides whether a wide weight's step runs inside the backward pass, so it cannot change inside an open
    window: the assignment is refused and the optimizer is left as it was; after step() it is accepted."""
    CpuAdam = _cpu_adam_class()
    w = torch.nn.Parameter(torch.randn(64))
    opt = CpuAdam([w])
    opt.log = []
    opt._fused[id(w)] = True                 # this window's step already ran inside the backward pass
    with pytest.raises(RuntimeError, match="between steps"):
        opt.gradient_clip_val = 1.0
    assert opt.gradient_clip_val == 0.0
    opt.gradient_clip_val = 0                # no change: accepted
    opt.step()
    assert opt.log == [] and not opt._fused
    opt.gradient_clip_val = 1.0
    assert opt.gradient_clip_val == 1.0
    with pytest.raises(ValueError):
        opt.gradient_clip_val = -1.0
    assert opt.gradient_clip_val == 1.0


def test_make_adam_reads_gradient_clip_val():
    """make_adam's reading of hparams.gradient_clip_val: passed to FusedAdam at world size 1; under torch.distributed
    left to the Trainer with a warning (FusedAdam does not clip there), so such a run still trains."""
    from types import SimpleNamespace
    from driving_dirty_b200.optim import follow_clipping
    assert follow_clipping(SimpleNamespace(), False) == 0.0 and follow_clipping(None, True) == 0.0
    assert follow_clipping(SimpleNamespace(gradient_clip_val=0.5), False) == 0.5
    assert follow_clipping(SimpleNamespace(gradient_clip_val=0), True) == 0.0
    with pytest.warns(UserWarning, match="torch.distributed"):
        assert follow_clipping(SimpleNamespace(gradient_clip_val=0.5), True) == 0.0
    with pytest.raises(ValueError):
        follow_clipping(SimpleNamespace(gradient_clip_val=-1), False)


def test_step_clips_what_it_applies():
    """One dd_grad_sumsq over every gradient the step applies -- all groups, an accumulation buffer in place of .grad,
    tensors without a gradient skipped -- before any Adam launch, and every launch takes the coefficient."""
    CpuAdam = _cpu_adam_class()
    w, b, frozen, s = (torch.nn.Parameter(torch.randn(n)) for n in (64, 8, 5, 3))
    opt = CpuAdam([{"params": [w, b]}, {"params": [frozen, s]}], gradient_clip_val=0.5)
    opt.log = []
    acc = torch.randn(64) * 10
    opt._passes[id(w)] = 2                   # w's window gathered in its accumulation buffer (world size 1, overlap)
    opt._acc_buf[id(w)] = acc
    b.grad, s.grad = torch.randn(8), torch.randn(3)
    opt.step()
    want = [acc.data_ptr(), b.grad.data_ptr(), s.grad.data_ptr()]
    assert opt.log[0] == ("clip", want)
    coef = 0.5 / (math.sqrt(sum(float((t.double() ** 2).sum()) for t in (acc, b.grad, s.grad))) + 1e-6)
    assert [e[:3] for e in opt.log[1:]] == [("adam", p.data_ptr(), g) for p, g in zip((w, b, s), want)]
    assert all(abs(e[3] - coef) < 1e-6 * coef for e in opt.log[1:])
    assert opt.last_grad_norm is not None and not opt._passes
    # clipping off: the same launches, no coefficient, no norm
    opt2 = CpuAdam([{"params": [w, b]}, {"params": [frozen, s]}])
    opt2.log = []
    opt2.step()
    assert all(e[0] == "adam" and e[3] is None for e in opt2.log) and opt2.last_grad_norm is None


def test_backward_hook_gives_up_the_fused_step():
    """Under clipping the wide weight's step cannot run inside the backward pass: at k = 1 ops.linear keeps the backward
    (autograd gets the gradient); at k > 1 the window's passes, the last one included, add into the buffer."""
    from driving_dirty_b200.optim import _BackwardHook
    CpuAdam = _cpu_adam_class()
    w = torch.nn.Parameter(torch.randn(16, 4))
    for clip, k, fusable, want in ((0.0, 1, True, True), (1.0, 1, True, False), (1.0, 1, False, False),
                                   (0.0, 2, True, True), (1.0, 2, True, True)):
        opt = CpuAdam([w], gradient_clip_val=clip, accumulate_grad_batches=k)
        hook = _BackwardHook(opt, opt.param_groups[0], w)
        assert hook.takes(fusable) == want, (clip, k, fusable)
    seen = []
    opt = CpuAdam([w], gradient_clip_val=1.0, accumulate_grad_batches=2)
    opt._window_backward = lambda g, p, dy, x, w_, dx, db, ws, n, fusable, impl: seen.append(fusable)
    _BackwardHook(opt, opt.param_groups[0], w)(None, None, None, None, None, None, 0, True, 0)
    assert seen == [False]


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from tests.test_grad_accumulation_cpu import _gloo_adam_class
    GlooAdam = _gloo_adam_class()
    params = [torch.nn.Parameter(torch.randn(64, 66)), torch.nn.Parameter(torch.randn(7))]
    res = {}
    try:
        GlooAdam(params, shard_min_numel=1024, gradient_clip_val=1.0)
        res["refused"] = False
    except NotImplementedError as e:
        res["refused"] = "gradient_clip_val" in str(e)
    opt = GlooAdam(params, shard_min_numel=1024, gradient_clip_val=0)
    res["off_accepted"] = opt.gradient_clip_val == 0.0
    try:
        opt.gradient_clip_val = 1.0
        res["setter_refused"] = False
    except NotImplementedError:
        res["setter_refused"] = opt.gradient_clip_val == 0.0
    q.put((rank, all(res.values()), res))
    dist.destroy_process_group()


def test_distributed_clipping_is_refused():
    """Clipping of the data-parallel form needs the norm of the rank-averaged gradient before the sharded update; until it
    has one, FusedAdam refuses gradient_clip_val under torch.distributed instead of clipping per-rank replicas."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 35500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=180) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(r[:2] for r in res) == [(0, True), (1, True)], res
