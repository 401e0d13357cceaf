"""Gradient norms in optim.FusedAdam (track_grad_norm), host logic on CPU with the device calls emulated: the flag's
validation and its changes between steps only, make_adam's reading of hparams.track_grad_norm, the modules' grad_norm()
keys and its deferral to the base class, grad_norms() refusing outside its valid range, and under gloo at world size 2 the
sharded bookkeeping (norm slots folded in rank order, the flat bucket staged once)."""
import os
import sys
from types import SimpleNamespace

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cpu_adam_class():
    from driving_dirty_b200.optim import FusedAdam

    class CpuAdam(FusedAdam):
        """World size 1 on CPU tensors: the per-tensor sums of squares computed in float64, the Adam launches skipped."""

        def _check_param(self, p):
            assert p.dtype == torch.float32 and p.is_contiguous()

        def _sumsq_each(self, grads, outs):
            for g, o in zip(grads, outs):
                o.copy_((g.double() ** 2).sum())

        def _launch_local(self, g, p, grad, coef=None):
            pass

    return CpuAdam


def test_track_grad_norm_value():
    from driving_dirty_b200.optim import track_grad_norm_value
    for off in (-1, 0, None, 0.0, -1.0):
        assert track_grad_norm_value(off) is False
    assert track_grad_norm_value(2) is True and track_grad_norm_value(2.0) is True
    for bad in (1, 3, float("inf"), "2", True, False, 2.5):
        with pytest.raises(ValueError, match="track_grad_norm=2"):
            track_grad_norm_value(bad)


def test_flag_changes_between_steps_only():
    CpuAdam = _cpu_adam_class()
    w = torch.nn.Parameter(torch.randn(16))
    opt = CpuAdam([w])
    assert opt.track_grad_norm == -1
    assert CpuAdam([w], track_grad_norm=2.0).track_grad_norm == 2
    with pytest.raises(ValueError):
        CpuAdam([w], track_grad_norm=1)
    opt._fused[id(w)] = True                 # this window's step already ran inside the backward pass
    with pytest.raises(RuntimeError, match="between steps"):
        opt.track_grad_norm = 2
    assert opt.track_grad_norm == -1
    opt.track_grad_norm = None               # no change: accepted
    opt.step()
    opt.track_grad_norm = 2
    assert opt.track_grad_norm == 2
    with pytest.raises(ValueError):
        opt.track_grad_norm = "inf"
    assert opt.track_grad_norm == 2


def test_make_adam_reads_track_grad_norm():
    from driving_dirty_b200.optim import follow_norm_tracking
    assert follow_norm_tracking(None) == -1 and follow_norm_tracking(SimpleNamespace()) == -1
    for off in (-1, 0, None):
        assert follow_norm_tracking(SimpleNamespace(track_grad_norm=off)) == -1
    assert follow_norm_tracking(SimpleNamespace(track_grad_norm=2)) == 2
    assert follow_norm_tracking(SimpleNamespace(track_grad_norm=2.0)) == 2
    for other in (1, 3, "inf"):
        with pytest.warns(UserWarning, match="left to Lightning"):
            assert follow_norm_tracking(SimpleNamespace(track_grad_norm=other)) == -1


def _module(opt_kind, track=2):
    from driving_dirty_b200.lightning_compat import FusedGradNorm, _MinimalLightningModule
    from driving_dirty_b200.optim import attach_optimizer

    class M(FusedGradNorm, _MinimalLightningModule):
        def __init__(self):
            super().__init__()
            self.fc1 = torch.nn.Linear(6, 4)
            self.frozen = torch.nn.Parameter(torch.randn(3), requires_grad=False)

    m = M()
    params = [p for p in m.parameters() if p.requires_grad]
    opt = _cpu_adam_class()(params, track_grad_norm=track) if opt_kind == "fused" else torch.optim.Adam(params)
    attach_optimizer(m, opt)
    m.fc1.weight.grad = torch.randn(4, 6)
    m.fc1.bias.grad = torch.randn(4)
    return m, opt


def test_grad_norm_keys_and_values():
    m, opt = _module("fused")
    out = m.grad_norm(2)
    assert set(out) == {"grad_2_norm_fc1.weight", "grad_2_norm_fc1.bias", "grad_2_norm_total"}
    w, b = m.fc1.weight.grad.double(), m.fc1.bias.grad.double()
    assert abs(float(out["grad_2_norm_fc1.weight"]) - float(w.norm())) < 1e-6 * float(w.norm())
    total = float((w.norm() ** 2 + b.norm() ** 2).sqrt())
    assert abs(float(out["grad_2_norm_total"]) - total) < 1e-6 * total
    assert all(torch.is_tensor(v) and v.dim() == 0 and v.dtype == torch.float32 for v in out.values())
    # keys follow norm_type as passed
    assert set(m.grad_norm(2.0)) == {"grad_2.0_norm_fc1.weight", "grad_2.0_norm_fc1.bias", "grad_2.0_norm_total"}


@pytest.mark.parametrize("kind,track,norm_type", [("torch", 2, 2), ("fused", -1, 2), ("fused", 2, 1)])
def test_grad_norm_defers_to_the_base_class(kind, track, norm_type):
    """--optimizer torch, tracking off, or a norm FusedAdam does not track: the base class's numbers (rounded floats)."""
    m, _ = _module(kind, track)
    out = m.grad_norm(norm_type)
    assert set(out) == {f"grad_{norm_type}_norm_fc1.weight", f"grad_{norm_type}_norm_fc1.bias",
                        f"grad_{norm_type}_norm_total"}
    assert all(isinstance(v, float) for v in out.values())


def test_grad_norms_refuses_outside_its_range():
    from driving_dirty_b200.optim import _BackwardHook
    CpuAdam = _cpu_adam_class()
    w, s = torch.nn.Parameter(torch.randn(16, 4)), torch.nn.Parameter(torch.randn(3))
    with pytest.raises(RuntimeError, match="track_grad_norm is off"):
        CpuAdam([w, s]).grad_norms()
    opt = CpuAdam([w, s], track_grad_norm=2, accumulate_grad_batches=3)
    with pytest.raises(RuntimeError, match="no gradient"):
        opt.grad_norms()
    # an open accumulation window: 1 of 3 passes
    opt._factor()
    opt._passes[id(w)] = 1
    opt._acc_buf[id(w)] = torch.randn(16, 4)
    with pytest.raises(RuntimeError, match="1 of its 3 backward passes"):
        opt.grad_norms()
    opt._passes[id(w)] = 3                   # complete (the last pass not fused): norms of the buffer
    s.grad = torch.randn(3)
    got = opt.grad_norms()
    assert abs(float(got[w]) - float(opt._acc_buf[id(w)].double().norm())) < 1e-5
    opt.step()
    after = opt.grad_norms()                  # after step(): the same numbers
    assert torch.equal(after[w], got[w]) and torch.equal(after["total"], got["total"])
    # the fused form: once the next window's backward pass has begun (stored gradients changed), they are gone
    opt2 = CpuAdam([w, s], track_grad_norm=2)
    w._dd_fused_update = _BackwardHook(opt2, opt2.param_groups[0], w)
    try:
        s.grad = torch.randn(3)
        opt2._fused[id(w)] = True
        opt2._present.add(id(w))
        opt2.grad_norms()
        opt2.step()
        opt2.grad_norms()
        s.grad = torch.randn(3)
        with pytest.raises(RuntimeError, match="next window"):
            opt2.grad_norms()
    finally:
        del w._dd_fused_update


def test_zero_grad_after_step_keeps_the_norms():
    """After step(), zero_grad() (to None or in place) clears gradients but starts no window: grad_norms() still returns
    the stepped window's norms, in the fused form too; a backward pass that writes stored gradients ends them."""
    from driving_dirty_b200.optim import _BackwardHook
    CpuAdam = _cpu_adam_class()
    w, s = torch.nn.Parameter(torch.randn(16, 4)), torch.nn.Parameter(torch.randn(3))
    for set_to_none in (True, False):
        opt = CpuAdam([w, s], track_grad_norm=2)
        w._dd_fused_update = _BackwardHook(opt, opt.param_groups[0], w)
        try:
            s.grad = torch.randn(3)
            opt._fused[id(w)] = True
            opt._present.add(id(w))
            got = opt.grad_norms()
            opt.step()
            opt.zero_grad(set_to_none=set_to_none)
            after = opt.grad_norms()
            assert torch.equal(after[s], got[s]) and torch.equal(after["total"], got["total"])
            s.grad = torch.randn(3) if set_to_none else s.grad.add_(1.0)
            with pytest.raises(RuntimeError, match="next window"):
                opt.grad_norms()
        finally:
            del w._dd_fused_update


def test_step_takes_the_stored_norms_when_first():
    """With tracking, step() takes the stored gradients' sums if grad_norms() did not; grad_norms() then reads them."""
    CpuAdam = _cpu_adam_class()
    w, s = torch.nn.Parameter(torch.randn(8)), torch.nn.Parameter(torch.randn(3))
    opt = CpuAdam([w, s], track_grad_norm=2)
    calls = []
    inner = opt._sumsq_each
    opt._sumsq_each = lambda g, o: (calls.append(len(g)), inner(g, o))
    w.grad, s.grad = torch.randn(8), torch.randn(3)
    opt.step()
    got = opt.grad_norms()
    assert calls == [2] and abs(float(got[s]) - float(s.grad.double().norm())) < 1e-6
    w.grad, s.grad = torch.randn(8), torch.randn(3)          # a new window of stored gradients
    got = opt.grad_norms()
    opt.step()
    assert calls == [2, 2] and abs(float(got[w]) - float(w.grad.double().norm())) < 1e-6


# ------------------------------------------------------------------------------------------------
# world size 2 under gloo
# ------------------------------------------------------------------------------------------------
def _gloo_norm_class():
    from tests.test_grad_accumulation_cpu import _gloo_adam_class
    Base = _gloo_adam_class()

    class GlooNormAdam(Base):
        def _launch_sharded(self, r, ctas_per_sm, norm=False):
            if norm:                            # this rank's shard sum of the rank mean, into its norm slot
                piece = self._symm["buf"][r["off"]: r["off"] + r["n"]].clone()
                every = [torch.empty_like(piece) for _ in range(self.world)]
                dist.all_gather(every, piece)
                mean = sum(every) / self.world
                self._slot_view()[self._norm_index[id(r["key"])]] = (mean[r["lo"]: r["hi"]].double() ** 2).sum()
            super()._launch_sharded(r, ctas_per_sm)

        def _sumsq_each_replicas(self, offs, numels, slots):
            self.flat_calls += 1
            buf = self._symm["buf"]
            every = [torch.empty_like(buf) for _ in range(self.world)]
            dist.all_gather(every, buf.clone())
            mean = sum(every) / self.world
            for o, n, i in zip(offs, numels, slots):
                self._slot_view()[i] = (mean[o: o + n].double() ** 2).sum()

        def _sumsq_each(self, grads, outs):
            for g, o in zip(grads, outs):
                o.copy_((g.double() ** 2).sum())

        def _slot_view(self):
            base, n = self._slots
            return self._mom[base: base + 2 * n].view(torch.float64)

    return GlooNormAdam


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from tests.test_grad_accumulation_cpu import _Stream, _backward
    torch.cuda.Stream = lambda *a, **k: _Stream()
    torch.cuda.current_stream = lambda *a, **k: _Stream()
    torch.cuda.stream = lambda s: s
    GlooNormAdam = _gloo_norm_class()

    res = {}
    g = torch.Generator().manual_seed(5)
    shapes = [(64, 66), (7,), (5,)]                            # one sharded wide weight, two flat-bucket tensors
    init = [torch.randn(s, generator=g) for s in shapes]
    grads = [[[[torch.randn(s, generator=g) for s in shapes] for _ in range(world)] for _ in range(2)] for _ in range(2)]
    for overlap in (True, False):
        params = [torch.nn.Parameter(t.clone()) for t in init]
        opt = GlooNormAdam(params, lr=1e-2, shard_min_numel=1024, overlap_backward=overlap, defer_join=False,
                           accumulate_grad_batches=2, track_grad_norm=2)
        opt.flat_calls = 0
        ok = True
        for w in range(2):
            opt.zero_grad()
            for j in range(2):
                _backward(params[0], grads[w][j][rank][0])
                for i in (1, 2):
                    params[i].grad = grads[w][j][rank][i].clone() if j == 0 else params[i].grad + grads[w][j][rank][i]
                if j == 0 and overlap:
                    try:
                        opt.grad_norms()
                        ok = False
                    except RuntimeError as e:
                        ok &= "1 of its 2 backward passes" in str(e)
            if overlap:
                got = opt.grad_norms()
            else:
                try:
                    opt.grad_norms()
                    ok = False
                except RuntimeError as e:
                    ok &= "only after step()" in str(e)
            opt.step()
            after = opt.grad_norms()
            if not overlap:
                got = after
            want = [sum(sum(grads[w][j][r][i] for j in range(2)) for r in range(world)).double() / world for i in range(3)]
            for i in range(3):
                ok &= abs(float(got[params[i]]) - float(want[i].norm())) < 1e-5 * float(want[i].norm())
                ok &= torch.equal(got[params[i]], after[params[i]])
            vec = torch.stack([got[p] for p in params] + [got["total"]])
            every = [torch.empty_like(vec) for _ in range(world)]
            dist.all_gather(every, vec)
            ok &= all(torch.equal(every[0], v) for v in every)     # the same bits on every rank
        res[f"overlap={overlap}"] = bool(ok) and opt.flat_calls == 2     # the flat bucket staged once per window
    q.put((rank, all(res.values()), res))
    dist.destroy_process_group()


def _flat_worker(rank, world, port, q):
    """No trainable wide weight (every tensor in the flat bucket), sharded and partly frozen (replicated) forms: every
    window's norms are that window's rank mean, and an in-place change of p.grad after grad_norms() (Lightning's clip)
    reaches the update exactly as without tracking."""
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from tests.test_grad_accumulation_cpu import _Stream
    torch.cuda.Stream = lambda *a, **k: _Stream()
    torch.cuda.current_stream = lambda *a, **k: _Stream()
    torch.cuda.stream = lambda s: s
    GlooNormAdam = _gloo_norm_class()
    res = {}
    g = torch.Generator().manual_seed(9)
    shapes = [(7,), (5,), (3,)]
    init = [torch.randn(s, generator=g) for s in shapes]
    windows = 3
    grads = [[[torch.randn(s, generator=g) for s in shapes] for _ in range(world)] for _ in range(windows)]
    for frozen in (False, True):
        runs = []
        for track in (False, True):
            params = [torch.nn.Parameter(t.clone()) for t in init]
            if frozen:
                params[2].requires_grad_(False)
            opt = GlooNormAdam(params, lr=1e-2, shard_min_numel=1 << 20, overlap_backward=True, defer_join=False,
                               track_grad_norm=2 if track else -1)
            opt.flat_calls = 0
            ok = True
            for w in range(windows):
                opt.zero_grad()
                live = [i for i in range(3) if not (frozen and i == 2)]
                for i in live:
                    params[i].grad = grads[w][rank][i].clone()
                if track:
                    got = opt.grad_norms()
                    want = [sum(grads[w][r][i] for r in range(world)).double() / world for i in live]
                    for i, m in zip(live, want):
                        ok &= abs(float(got[params[i]]) - float(m.norm())) < 1e-5 * float(m.norm())
                    ok &= (params[2] in got) != frozen
                    vec = torch.stack([got[params[i]] for i in live] + [got["total"]])
                    every = [torch.empty_like(vec) for _ in range(world)]
                    dist.all_gather(every, vec)
                    ok &= all(torch.equal(every[0], v) for v in every)
                for i in live:                         # what Lightning's clip does to p.grad before optimizer.step()
                    params[i].grad.mul_(0.5)
                opt.step()
                if track:
                    after = opt.grad_norms()             # after step(): the window's norms, now of the clipped gradients
                    for i, m in zip(live, want):
                        ok &= abs(float(after[params[i]]) - 0.5 * float(m.norm())) < 1e-5 * float(m.norm())
            runs.append(([p.detach().clone() for p in params], ok))
        (w_off, _), (w_on, ok) = runs
        res[f"frozen={frozen}"] = ok and all(torch.equal(a, b) for a, b in zip(w_off, w_on))
    q.put((rank, all(res.values()), res))
    dist.destroy_process_group()


def test_flat_only_windows_gloo():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 38500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_flat_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=180) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(r[:2] for r in res) == [(0, True), (1, True)], res


def test_sharded_norms_gloo():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 36500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=180) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(r[:2] for r in res) == [(0, True), (1, True)], res
