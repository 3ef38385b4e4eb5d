#!/usr/bin/env python
"""Channel concatenation and the U-Net on one B200: dfb_concat_channels_fwd / _bwd at the skip connections of a batch-256
U-Net decoder, each beside dfb_copy of the same byte count (the device's plain copy, a yardstick), timed alternately in the
same run against the minimum bytes; then the unet workload's captured training step (Adam, CapturedStep) in images/s.
Event timing and L2 flush are opbench.py's.

    python scripts/unet_bench.py [--batch 256] [--iters 20] [--mode tf32] [--steps 30] [--out DIR]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import deepflows_b200  # noqa: E402,F401
import workloads  # noqa: E402
from opbench import event_timer  # noqa: E402

# (up channels, skip channels, spatial size): the three skip connections of unet(widths=(32, 64, 128, 256)) at 64x64
CAT_SHAPES = [(32, 32, 64), (64, 64, 32), (128, 128, 16)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi failed)"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--mode", default="tf32")
    ap.add_argument("--steps", type=int, default=30, help="timed U-Net steps")
    ap.add_argument("--out", default=None, help="directory for unet_bench.json")
    args = ap.parse_args()
    from DeepFlows import backend_api, nn
    from DeepFlows.tensor import Tensor
    from DeepFlows.cuda_graph import CapturedStep
    import DeepFlows
    dev = backend_api.cuda()
    if not dev.enabled() or dev.device_count() == 0:
        raise SystemExit("unet_bench: no CUDA device (this measurement has no CPU variant)")
    m = dev.mod
    backend_api.set_precision(args.mode)
    flush = m.Array(64 << 20)  # 256 MB > 126 MB L2
    time_it = event_timer(m, args.iters, flush)
    rng = np.random.RandomState(0)
    gpu = card()
    n = args.batch
    print("card (name, power limit, max SM clock): %s; mode %s, batch %d, L2 flushed before every timed call" % (gpu, args.mode, n))
    res = {"card": gpu, "mode": args.mode, "batch": n, "concat": []}

    def dev_rand(k):
        a = m.Array(k)
        m.from_numpy(rng.randn(k).astype(np.float32), a)
        return a

    print("\nconcat of (up, skip) channels-last; GB/s against the minimum bytes 8 * |y| (read every element once, write it once),")
    print("beside dfb_copy of 4 * |y| bytes; median of 3 alternated runs of %d timed calls each" % args.iters)
    print("%-24s %-4s %10s %9s %10s %9s" % ("shape", "pass", "cat us", "cat GB/s", "copy us", "copy GB/s"))
    for cu, cs, hw in CAT_SHAPES:
        rows = n * hw * hw
        c = cu + cs
        up, skip, y, gy, dup, dskip = (dev_rand(rows * cu), dev_rand(rows * cs), m.Array(rows * c), dev_rand(rows * c),
                                       m.Array(rows * cu), m.Array(rows * cs))
        src, dst = dev_rand(rows * c), m.Array(rows * c)
        nbytes = 8.0 * rows * c
        calls = {"fwd": lambda: m.concat_channels_fwd([up, skip], [cu, cs], y, rows),
                 "bwd": lambda: m.concat_channels_bwd(gy, [dup, dskip], [cu, cs], rows)}
        # the kernels copy: check them once against numpy before timing
        calls["fwd"]()
        calls["bwd"]()
        ynp = m.to_numpy(y, (rows, c), (c, 1), 0)
        assert np.array_equal(ynp[:, :cu], m.to_numpy(up, (rows, cu), (cu, 1), 0))
        assert np.array_equal(ynp[:, cu:], m.to_numpy(skip, (rows, cs), (cs, 1), 0))
        assert np.array_equal(m.to_numpy(dskip, (rows, cs), (cs, 1), 0), m.to_numpy(gy, (rows, c), (c, 1), 0)[:, cu:])
        shape = "%dx%dx%dx(%d+%d)" % (n, hw, hw, cu, cs)
        for pas in ("fwd", "bwd"):
            a, b = [], []
            for _ in range(3):   # alternate the two calls so that both see the same clocks
                a.append(time_it(calls[pas]))
                b.append(time_it(lambda: m.copy(src, dst, rows * c)))
            ta, tb = float(np.median(a)), float(np.median(b))
            print("%-24s %-4s %10.1f %9.0f %10.1f %9.0f" % (shape, pas, ta, nbytes / ta / 1e3, tb, nbytes / tb / 1e3))
            res["concat"].append({"shape": shape, "pass": pas, "cat_us": ta, "cat_gbs": nbytes / ta / 1e3, "copy_us": tb,
                                  "copy_gbs": nbytes / tb / 1e3, "cat_runs_us": a, "copy_runs_us": b})
        del up, skip, y, gy, dup, dskip, src, dst

    # the U-Net's captured training step
    df = workloads.namespace(DeepFlows)
    np.random.seed(0)
    model = workloads.unet(df, "cuda")
    opt = df.optim.Adam(model.parameters(), lr=1e-3)
    crit = nn.MSELoss()
    x = Tensor(backend_api.Btensor(rng.randn(n, 3, 64, 64).astype(np.float32), device=dev))
    target = Tensor(backend_api.Btensor(np.tanh(rng.randn(n, 3, 64, 64)).astype(np.float32), device=dev))

    def step_fn():
        loss = crit(model(x), target)
        opt.zero_grad()
        loss.backward()
        opt.step()
        return loss

    step = CapturedStep(step_fn, device=dev, warmup=1)
    for _ in range(5):
        step()
    dev.synchronize()
    e0, e1 = m.event_create(), m.event_create()
    m.event_record(e0)
    for _ in range(args.steps):
        loss = step()
    m.event_record(e1)
    m.event_synchronize(e1)
    ms = m.event_elapsed_ms(e0, e1) / args.steps
    assert step.captured and np.isfinite(loss.data.numpy()).all()
    step.destroy()
    print("\nunet training step (widths 32-64-128-256, batch %d, 64x64x3 input, MSE, Adam, captured, %s): %.3f ms/step, %.0f images/s"
          % (n, args.mode, ms, n / ms * 1e3))
    res["unet"] = {"ms_per_step": ms, "images_per_s": n / ms * 1e3, "steps": args.steps}
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "unet_bench.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
