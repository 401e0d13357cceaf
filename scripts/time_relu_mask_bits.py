"""The four encoder kernels whose ReLU mask can travel as sign words (one uint32 per pixel, bit c = stored bf16 activation of
channel c > 0) instead of the 64-byte bf16 activation, at the bench shape (B = 32 scenes, 256 x 1836 mosaic, raw-byte
views into c1): c1 forward and c2 forward (plain / also writing the sign words), c2 and c3 input gradients (mask from the
activation / from the sign words).  CUDA events over ITERS launches per form, the two forms alternating, ROUNDS rounds,
after a warm-up; algorithmic bytes and GB/s, against the copy bandwidth of a torch copy measured in the same run.  Every
buffer a launch touches is 60-960 MB and one launch's working set is 1-3 GB, far beyond the 126 MB L2, so no cache flush is
needed between launches.  The two forms' outputs are compared bit for bit."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from driving_dirty_b200 import _lib  # noqa: E402
from driving_dirty_b200._lib import call, stream_ptr  # noqa: E402

ITERS, ROUNDS = int(os.environ.get("ITERS", 20)), int(os.environ.get("ROUNDS", 3))
B, H, W = 32, 256, 306
BF = _lib.DD_BF16


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                        "--format=csv"], capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name()


def event_ms(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    dev = torch.device("cuda")
    print(f"GPU (nvidia-smi, same run):\n{gpu_info()}")
    Wm, st = 6 * W, stream_ptr()
    H3, W3 = (H - 1) // 2 + 1, (Wm - 1) // 2 + 1
    g = torch.Generator(device=dev).manual_seed(1)
    views = torch.randint(0, 256, (B, 6, 3, H, W), dtype=torch.uint8, device=dev, generator=g)
    w1 = (torch.rand(32, 3, 3, 3, device=dev, generator=g) - 0.5) * 0.4
    w2 = (torch.rand(32, 32, 3, 3, device=dev, generator=g) - 0.5) * 0.12
    w3 = (torch.rand(32, 32, 3, 3, device=dev, generator=g) - 0.5) * 0.12
    bias = (torch.rand(32, device=dev, generator=g) - 0.5) * 0.2
    act = lambda: torch.empty(B, H, Wm, 32, dtype=torch.bfloat16, device=dev)  # noqa: E731
    bits = lambda: torch.empty(B, H, Wm, dtype=torch.int32, device=dev)  # noqa: E731
    a1, a1b, a2, a2b = act(), act(), act(), act()
    s1, s2 = bits(), bits()
    da2 = (torch.randn(B, H, Wm, 32, device=dev, generator=g) * 0.1).to(torch.bfloat16)
    da3 = (torch.randn(B, H3, W3, 32, device=dev, generator=g) * 0.1).to(torch.bfloat16)
    da1, da1b, da2o, da2ob = act(), act(), act(), act()
    p = lambda t: t.data_ptr()  # noqa: E731

    kernels = {
        "c1 fwd (u8 views)": {
            "mask": lambda: call("dd_conv_c1_fwd", p(views), 3, p(w1), p(bias), p(a1), BF, B, H, Wm, 2, st),
            "bits": lambda: call("dd_conv_c1_fwd_bits", p(views), 3, p(w1), p(bias), p(a1b), p(s1), BF, B, H, Wm, 2, st)},
        "c2 fwd (s1)": {
            "mask": lambda: call("dd_conv3x3_c32_fwd", p(a1), p(w2), p(bias), p(a2), BF, B, H, Wm, 1, 2, st),
            "bits": lambda: call("dd_conv3x3_c32_fwd_bits", p(a1), p(w2), p(bias), p(a2b), p(s2), BF, B, H, Wm, 1, 2, st)},
        "c2 dgrad (s1)": {
            "mask": lambda: call("dd_conv3x3_c32_dgrad", p(da2), p(w2), p(a1), p(da1), BF, B, H, Wm, 1, 2, st),
            "bits": lambda: call("dd_conv3x3_c32_dgrad_bits", p(da2), p(w2), p(s1), p(da1b), BF, B, H, Wm, 1, 2, st)},
        "c3 dgrad (s2)": {
            "mask": lambda: call("dd_conv3x3_c32_dgrad", p(da3), p(w3), p(a2), p(da2o), BF, B, H, Wm, 2, 2, st),
            "bits": lambda: call("dd_conv3x3_c32_dgrad_bits", p(da3), p(w3), p(s2), p(da2ob), BF, B, H, Wm, 2, 2, st)},
    }
    # algorithmic bytes: every input read once, every output written once
    A, A3, S, V = a1.numel() * 2, da3.numel() * 2, s1.numel() * 4, views.numel()
    nbytes = {"c1 fwd (u8 views)": (V + A, V + A + S), "c2 fwd (s1)": (2 * A, 2 * A + S),
              "c2 dgrad (s1)": (3 * A, 2 * A + S), "c3 dgrad (s2)": (A3 + 2 * A, A3 + A + S)}

    for name, forms in kernels.items():          # in pipeline order: c1 -> c2 -> dgrads read what the forwards wrote
        forms["mask"](); forms["bits"]()
    torch.cuda.synchronize()
    v16 = lambda t: t.view(torch.int16)  # noqa: E731
    shifts = torch.arange(32, device=dev, dtype=torch.int64)
    pack = lambda a: ((a > 0).to(torch.int64) << shifts).sum(-1)  # noqa: E731
    checks = {"a1": torch.equal(v16(a1), v16(a1b)), "a2": torch.equal(v16(a2), v16(a2b)),
              "a1 sign words": torch.equal(s1.to(torch.int64) & 0xFFFFFFFF, pack(a1)),
              "a2 sign words": torch.equal(s2.to(torch.int64) & 0xFFFFFFFF, pack(a2)),
              "da1": torch.equal(v16(da1), v16(da1b)), "da2": torch.equal(v16(da2o), v16(da2ob))}
    print("bit-identical between the forms: " + ", ".join(f"{k} {'yes' if v else 'NO'}" for k, v in checks.items()))
    print(f"share of zero activations: a1 {float((a1 == 0).float().mean()):.2f}, a2 {float((a2 == 0).float().mean()):.2f}")

    src = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    for _ in range(3):
        dst.copy_(src)
    copy_ms = min(event_ms(lambda: dst.copy_(src), ITERS) for _ in range(ROUNDS))
    roof = 2 * src.numel() / copy_ms * 1e-6
    print(f"copy bandwidth (torch copy of 1 GiB, read + write): {roof:.0f} GB/s")
    del src, dst

    print(f"B {B}, mosaic {H} x {Wm}; {ITERS} launches per timing, {ROUNDS} rounds, forms alternating; min over rounds")
    total = {"mask": 0.0, "bits": 0.0}
    for name, forms in kernels.items():
        for form in ("mask", "bits"):
            for _ in range(3):
                forms[form]()
        times = {"mask": [], "bits": []}
        for _ in range(ROUNDS):
            for form in ("mask", "bits"):
                times[form].append(event_ms(forms[form], ITERS))
        for i, form in enumerate(("mask", "bits")):
            t, nb = min(times[form]), nbytes[name][i]
            total[form] += t
            label = {"mask": "activation" if "dgrad" in name else "plain", "bits": "sign words"}[form]
            print(f"  {name:18s} {label:10s} {t:.3f} ms (rounds {', '.join(f'{x:.3f}' for x in times[form])})  "
                  f"{nb / 1e9:.3f} GB -> {nb / t * 1e-6:.0f} GB/s = {nb / t * 1e-6 / roof:.0%} of copy")
    print(f"four kernels: {total['mask']:.3f} ms with the activation masks, {total['bits']:.3f} ms with sign words "
          f"({total['mask'] - total['bits']:+.3f} ms)")


if __name__ == "__main__":
    main()
