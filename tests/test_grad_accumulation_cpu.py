"""Gradient accumulation in optim.FusedAdam's data-parallel form, host logic on CPU: a world-size-2 gloo run in which the
window bookkeeping (overwrite on the first pass, accumulate on the later ones, the sharded update launched on pass k, a
partial window, the refusal of pass k + 1, zero_grad discarding an unfinished window) runs unchanged and only the device
touch points are emulated, as in test_distributed_cpu.py; and make_adam's reading of hparams.accumulate_grad_batches."""
import os
import sys
from types import SimpleNamespace

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _Stream:
    """Stand-in for the side stream of overlap_backward: work "on" it runs at once."""

    def wait_stream(self, other):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def _gloo_adam_class():
    from driving_dirty_b200.optim import FusedAdam, shard_bounds

    class _Handle:
        def barrier(self, channel=0):
            dist.barrier()

    class GlooAdam(FusedAdam):
        launches = 0

        def _check_param(self, p):
            assert p.dtype == torch.float32 and p.is_contiguous()

        def _alloc_symmetric(self, numel, device, multicast):
            return torch.empty(numel, dtype=torch.float32), _Handle(), [0] * self.world, 0

        def _alloc_moments(self, numel, device):
            buf = torch.zeros(numel, dtype=torch.float32)

            def peer(rk):
                t = buf.clone()
                dist.broadcast(t, src=rk)
                return t
            return buf, peer

        def _launch_sharded(self, r, ctas_per_sm):
            # reduce (mean of the replicas) + torch.optim.Adam's arithmetic on this rank's shard + all-gather
            GlooAdam.launches += 1
            sy = self._symm
            buf, total, off, lo, hi = sy["buf"], sy["total"], r["off"], r["lo"], r["hi"]
            parts = None
            for rk in range(self.world):
                lo_k, hi_k = shard_bounds(r["n"], self.world, rk)
                piece = buf[off + lo_k: off + hi_k].clone()
                got = [torch.empty_like(piece) for _ in range(self.world)] if rk == self.rank else None
                dist.gather(piece, got, dst=rk)
                if rk == self.rank:
                    parts = got
            g = sum(parts) / self.world
            st = self._shard_state(r)
            st["step"] += 1
            lr, b1, b2, eps, wd = self._hyper()
            w = buf[total + off + lo: total + off + hi]
            if wd:
                g = g + wd * w
            st["exp_avg"].lerp_(g, 1 - b1)
            st["exp_avg_sq"].mul_(b2).addcmul_(g, g, value=1 - b2)
            bc1, bc2 = 1 - b1 ** st["step"], 1 - b2 ** st["step"]
            w.sub_((lr / bc1) * st["exp_avg"] / (st["exp_avg_sq"].sqrt() / bc2 ** 0.5 + eps))
            for rk in range(self.world):
                lo_k, hi_k = shard_bounds(r["n"], self.world, rk)
                dist.broadcast(buf[total + off + lo_k: total + off + hi_k], src=rk)

        def _launch_local(self, g, p, grad):
            st = self._state(p, p.numel(), p.device)
            st["step"] += 1
            lr, b1, b2, eps, wd = self._hyper()
            gr = grad + wd * p.data if wd else grad
            st["exp_avg"].lerp_(gr.reshape(-1), 1 - b1)
            st["exp_avg_sq"].mul_(b2).addcmul_(gr.reshape(-1), gr.reshape(-1), value=1 - b2)
            bc1, bc2 = 1 - b1 ** st["step"], 1 - b2 ** st["step"]
            p.data.sub_(((lr / bc1) * st["exp_avg"] / (st["exp_avg_sq"].sqrt() / bc2 ** 0.5 + eps)).view_as(p))

    return GlooAdam


def _backward(p, grad):
    """What ops.linear's backward does with a sharded weight: ask whether to accumulate, write (or add), signal."""
    acc = p._dd_grad_begin()
    if acc:
        p._dd_grad_buffer.add_(grad)         # dd_linear_wgrad_acc: old + this pass's gradient
    else:
        p._dd_grad_buffer.copy_(grad)        # dd_linear_wgrad
    p._dd_grad_ready()
    return acc


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.cuda.Stream = lambda *a, **k: _Stream()              # overlap_backward's side stream, emulated
    torch.cuda.current_stream = lambda *a, **k: _Stream()
    torch.cuda.stream = lambda s: s
    GlooAdam = _gloo_adam_class()
    res = {}
    g = torch.Generator().manual_seed(5)
    shapes = [(64, 66), (7,)]                                  # one sharded wide weight, one flat-bucket tensor
    init = [torch.randn(s, generator=g) for s in shapes]
    # grads[window][pass][rank][tensor]
    grads = [[[[torch.randn(s, generator=g) for s in shapes] for _ in range(world)] for _ in range(3)] for _ in range(4)]

    def run(overlap, plan):
        """plan: passes per window; the factor is 2 except where a window lists (passes, k)."""
        params = [torch.nn.Parameter(t.clone()) for t in init]
        opt = GlooAdam(params, lr=1e-2, weight_decay=0.01, shard_min_numel=1024, overlap_backward=overlap,
                       defer_join=False, accumulate_grad_batches=2)
        ref = [t.clone().requires_grad_(True) for t in init]
        ropt = torch.optim.Adam(ref, lr=1e-2, weight_decay=0.01)
        log = []
        for w, item in enumerate(plan):
            passes, k = item if isinstance(item, tuple) else (item, 2)
            opt.accumulate_grad_batches = k
            opt.zero_grad()
            GlooAdam.launches = 0
            for j in range(passes):
                acc = _backward(params[0], grads[w][j][rank][0])
                params[1].grad = grads[w][j][rank][1].clone() if j == 0 else params[1].grad + grads[w][j][rank][1]
                log.append((acc, GlooAdam.launches, id(params[0]) in opt._launched))
            opt.step()
            for i, p in enumerate(ref):
                p.grad = sum(sum(grads[w][j][r][i] for j in range(passes)) for r in range(world)) / world
            ropt.step()
        err = max(float((a.detach() - b.detach()).abs().max()) for a, b in zip(params, ref))
        return err, log, opt, params

    # full windows of k = 2, then a window of k = 3, then a partial window (2 of 3 passes), overlap off and on
    for overlap in (False, True):
        err, log, _, _ = run(overlap, [2, 2, (3, 3), (2, 3)])
        accs = [a for a, _, _ in log]
        launched = [(n, lz) for _, n, lz in log]
        res[f"err_{overlap}"] = err
        res[f"acc_{overlap}"] = accs == [0, 1, 0, 1, 0, 1, 1, 0, 1]
        if overlap:    # the sharded update leaves from the window's last pass only: none from passes 1 .. k-1
            res["launch_on_k"] = launched == [(0, False), (1, True), (0, False), (1, True), (0, False), (0, False),
                                              (1, True), (0, False), (0, False)]
        else:
            res["no_launch_in_backward"] = all(n == 0 and not lz for n, lz in launched)

    # pass k + 1 of a window is refused before anything is written, naming the flag
    params = [torch.nn.Parameter(t.clone()) for t in init]
    opt = GlooAdam(params, lr=1e-2, shard_min_numel=1024, accumulate_grad_batches=2)
    _backward(params[0], grads[0][0][rank][0])
    _backward(params[0], grads[0][1][rank][0])
    try:
        params[0]._dd_grad_begin()
        res["refused"] = False
    except RuntimeError as e:
        res["refused"] = "accumulate_grad_batches=2" in str(e)
    try:
        params[0]._dd_grad_ready()
        res["refused_ready"] = False
    except RuntimeError as e:
        res["refused_ready"] = "accumulate_grad_batches=2" in str(e)
    opt.step()
    res["window_reset_by_step"] = params[0]._dd_grad_begin() == 0

    # zero_grad discards an unfinished window: the next pass overwrites the replica again
    params = [torch.nn.Parameter(t.clone()) for t in init]
    opt = GlooAdam(params, lr=1e-2, shard_min_numel=1024, accumulate_grad_batches=2)
    _backward(params[0], torch.full(shapes[0], 1e3))
    opt.zero_grad()
    res["zero_grad_resets"] = _backward(params[0], grads[1][0][rank][0]) == 0 and \
        _backward(params[0], grads[1][1][rank][0]) == 1
    params[1].grad = grads[1][0][rank][1] + grads[1][1][rank][1]
    opt.step()
    ref = [t.clone().requires_grad_(True) for t in init]
    ropt = torch.optim.Adam(ref, lr=1e-2)
    for i, p in enumerate(ref):
        p.grad = sum(grads[1][0][r][i] + grads[1][1][r][i] for r in range(world)) / world
    ropt.step()
    res["zero_grad_err"] = max(float((a.detach() - b.detach()).abs().max()) for a, b in zip(params, ref))

    # a {epoch: factor} schedule is read at the first pass of each window
    params = [torch.nn.Parameter(t.clone()) for t in init]
    opt = GlooAdam(params, lr=1e-2, shard_min_numel=1024, accumulate_grad_batches={0: 1, 2: 3})
    epoch = [0]
    opt.current_epoch = lambda: epoch[0]
    _backward(params[0], grads[0][0][rank][0])
    ks = [opt._window_k]
    opt.step()
    epoch[0] = 2
    _backward(params[0], grads[0][0][rank][0])
    epoch[0] = 0                                               # changes inside a window do not reach it
    _backward(params[0], grads[0][1][rank][0])
    ks.append(opt._window_k)
    opt.step()
    res["schedule"] = ks == [1, 3]

    ok = all(v is True for k, v in res.items() if not k.startswith(("err", "zero_grad_err"))) and \
        res["err_False"] < 1e-6 and res["err_True"] < 1e-6 and res["zero_grad_err"] < 1e-6
    q.put((rank, ok, res))
    dist.destroy_process_group()


def test_fused_adam_accumulation_windows_two_ranks():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 33500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=180) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(r[:2] for r in res) == [(0, True), (1, True)], res


def test_accumulation_factor_int_and_schedule():
    from driving_dirty_b200.optim import accumulation_factor
    assert accumulation_factor(1) == 1 and accumulation_factor(4) == 4
    sched = {0: 1, 3: 2, 6: 4}
    assert [accumulation_factor(sched, e) for e in range(8)] == [1, 1, 1, 2, 2, 2, 4, 4]
    assert accumulation_factor({2: 3}, 0) == 1                 # before the first key: one pass per step
    for bad in (0, -1, 1.5, True, {0: 0}):
        with pytest.raises(ValueError):
            accumulation_factor(bad)


def test_make_adam_reads_accumulate_grad_batches():
    """make_adam hands FusedAdam the Namespace's accumulate_grad_batches (an int or a {epoch: factor} dict, resolved
    against the module's current_epoch); without the attribute the factor is 1."""
    from driving_dirty_b200.optim import follow_accumulation, accumulation_factor

    class Opt:
        pass

    for acc, epoch, want in ((None, 0, 1), (4, 0, 4), ({0: 1, 2: 3}, 1, 1), ({0: 1, 2: 3}, 5, 3)):
        hp = SimpleNamespace(lr=1e-3) if acc is None else SimpleNamespace(lr=1e-3, accumulate_grad_batches=acc)
        module = SimpleNamespace(hparams=hp, current_epoch=epoch)
        opt = Opt()
        follow_accumulation(opt, module)
        assert accumulation_factor(opt.accumulate_grad_batches, opt.current_epoch()) == want
    with pytest.raises(ValueError):
        follow_accumulation(Opt(), SimpleNamespace(hparams=SimpleNamespace(accumulate_grad_batches=0), current_epoch=0))
