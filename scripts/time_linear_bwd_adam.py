"""The backward pass + Adam step of the two wide FC layers of the RoadMapBCE training step, at the bench shapes: the three
unfused launches (dd_linear_dgrad + dd_linear_wgrad + dd_adam_step) against the one fused launch (dd_linear_bwd_adam).
CUDA events over ITERS iterations per form, the two forms alternating, ROUNDS rounds; algorithmic bytes and GB/s against
MEASURED_PEAKS.json (hbm_gbs) when present; the outputs of the two forms (dx, db, W, m, v) compared bit for bit."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from driving_dirty_b200 import _lib  # noqa: E402
from driving_dirty_b200._lib import call, stream_ptr  # noqa: E402

ITERS, ROUNDS = int(os.environ.get("ITERS", 20)), int(os.environ.get("ROUNDS", 3))
SHAPES = {"fc1": (32, 256, 940032, torch.bfloat16), "head": (32, 640000, 128, torch.float32)}   # B, N, K, dx dtype
LR, B1, B2, EPS, WD = 1e-3, 0.9, 0.999, 1e-8, 0.0


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name()


def main():
    dev = torch.device("cuda")
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peak = float(json.load(f)["hbm_gbs"])
    except (OSError, KeyError, ValueError):
        peak = None
    print(f"GPU: {gpu_info()}   copy bandwidth (MEASURED_PEAKS.json): {peak if peak else 'not found'} GB/s")
    g = torch.Generator(device=dev).manual_seed(1)
    for name, (B, N, K, dxt) in SHAPES.items():
        esz = torch.finfo(dxt).bits // 8
        x = torch.randn(B, K, device=dev, generator=g)
        dy = torch.randn(B, N, device=dev, generator=g) * 1e-3
        w0 = torch.randn(N, K, device=dev, generator=g) * 0.01
        m0 = torch.randn(N, K, device=dev, generator=g) * 1e-4
        v0 = torch.rand(N, K, device=dev, generator=g) * 1e-6
        n_ws = int(_lib.load().dd_linear_workspace_bytes(B, N, K))
        ws = torch.empty(n_ws, dtype=torch.uint8, device=dev)
        dw = torch.empty(N, K, device=dev)
        forms = {}
        for form in ("unfused", "fused"):
            forms[form] = dict(w=w0.clone(), m=m0.clone(), v=v0.clone(), dx=torch.empty(B, K, dtype=dxt, device=dev),
                               db=torch.empty(N, device=dev), step=0)

        def run(form):
            s = forms[form]
            s["step"] += 1
            code = _lib.dtype_code(dxt)
            if form == "fused":
                call("dd_linear_bwd_adam", dy.data_ptr(), x.data_ptr(), s["w"].data_ptr(), s["m"].data_ptr(), s["v"].data_ptr(),
                     s["dx"].data_ptr(), code, s["db"].data_ptr(), ws.data_ptr(), n_ws, B, N, K, LR, B1, B2, EPS, WD, s["step"],
                     stream_ptr())
            else:
                call("dd_linear_dgrad", dy.data_ptr(), s["w"].data_ptr(), s["dx"].data_ptr(), code, ws.data_ptr(), n_ws, B, N, K,
                     _lib.IMPL_TCGEN05, stream_ptr())
                call("dd_linear_wgrad", dy.data_ptr(), x.data_ptr(), _lib.DD_F32, dw.data_ptr(), s["db"].data_ptr(), B, N, K,
                     _lib.IMPL_TCGEN05, stream_ptr())
                call("dd_adam_step", s["w"].data_ptr(), dw.data_ptr(), s["m"].data_ptr(), s["v"].data_ptr(), N * K, LR, B1, B2,
                     EPS, WD, s["step"], 1.0, stream_ptr())

        # one step each from the same state, compared bit for bit
        run("unfused"); run("fused")
        torch.cuda.synchronize()
        same = {k: torch.equal(forms["unfused"][k], forms["fused"][k]) for k in ("dx", "db", "w", "m", "v")}
        print(f"{name}: B {B} N {N} K {K} dx {str(dxt).split('.')[-1]}; outputs of one step bit-identical: "
              + ", ".join(f"{k} {'yes' if v else 'NO'}" for k, v in same.items()))
        # algorithmic bytes: the 4-byte W / dW / m / v arrays, plus x, dy, dx, db
        small = 4 * B * K + 4 * B * N + esz * B * K + 4 * N
        nbytes = {"unfused": 36 * N * K + small + 4 * B * N, "fused": 24 * N * K + small + 4 * B * N}  # dy read twice by each
        times = {"unfused": [], "fused": []}
        for form in ("unfused", "fused"):       # warm-up
            for _ in range(3):
                run(form)
        for _ in range(ROUNDS):
            for form in ("unfused", "fused"):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record()
                for _ in range(ITERS):
                    run(form)
                e1.record()
                torch.cuda.synchronize()
                times[form].append(e0.elapsed_time(e1) / ITERS)
        for form in ("unfused", "fused"):
            t = min(times[form])
            gbs = nbytes[form] / t * 1e-6
            share = f" = {gbs / peak:.0%} of copy bandwidth" if peak else ""
            print(f"  {form:8s} {t:.3f} ms (rounds: {', '.join(f'{x:.3f}' for x in times[form])})  "
                  f"{nbytes[form] / 1e9:.2f} GB algorithmic -> {gbs:.0f} GB/s{share}")
        print(f"  saving {min(times['unfused']) - min(times['fused']):.3f} ms per step")
        del forms, dw, w0, m0, v0
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
