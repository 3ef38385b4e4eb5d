#!/usr/bin/env python
"""Decoder layers on one B200: ConvTranspose2d forward / backward-input / backward-weight at batch-256 generator shapes, each
beside the mirrored Conv2d call (same entry point, operands allocated as a Conv2d layer holds them), timed alternately in
the same run; Upsample nearest / bilinear forward / backward against their minimum bytes; the dcgan_generator workload's
captured training step (Adam, CapturedStep) in images/s. Event timing and L2 flush are opbench.py's.

    python scripts/decoder_bench.py [--batch 256] [--iters 20] [--mode tf32] [--out DIR]
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

# (in, out, input size, k, stride, padding, output_padding)
CT_SHAPES = [(256, 128, 8, 4, 2, 1, 0), (128, 64, 16, 4, 2, 1, 0), (64, 32, 32, 4, 2, 1, 0),
             (256, 128, 8, 3, 2, 1, 1), (128, 64, 16, 3, 2, 1, 1), (64, 32, 32, 3, 2, 1, 1)]
UP_SHAPES = [(64, 32, 2), (64, 64, 2)]   # (channels, input size, scale)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi failed)"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--mode", default="tf32")
    ap.add_argument("--steps", type=int, default=50, help="timed generator steps")
    ap.add_argument("--out", default=None, help="directory for decoder_bench.json")
    args = ap.parse_args()
    from DeepFlows import backend_api, nn, tensor
    from DeepFlows.tensor import Tensor
    from DeepFlows.cuda_graph import CapturedStep
    import DeepFlows
    dev = backend_api.cuda()
    if not dev.enabled() or dev.device_count() == 0:
        raise SystemExit("decoder_bench: no CUDA device (this measurement has no CPU variant)")
    m = dev.mod
    mode = {"fp32": m.MODE_FP32, "tf32": m.MODE_TF32}[args.mode]
    backend_api.set_precision(args.mode)
    flush = m.Array(64 << 20)  # 256 MB > 126 MB L2
    time_it = event_timer(m, args.iters, flush)
    rng = np.random.RandomState(0)
    gpu = card()
    print("card (name, power limit, max SM clock): %s; mode %s, batch %d, L2 flushed before every timed call" % (gpu, args.mode, args.batch))
    res = {"card": gpu, "mode": args.mode, "batch": args.batch, "conv_transpose": [], "upsample": []}

    def dev_rand(n):
        a = m.Array(n)
        m.from_numpy(rng.randn(n).astype(np.float32), a)
        return a

    def ws_for(geom):
        n_floats = m.conv2d_workspace_floats(*geom)
        return (m.Array(n_floats), n_floats) if n_floats else (None, 0)

    n = args.batch
    print("\nConvTranspose2d (in->out, size, k/s/p/op) vs the mirrored Conv2d call; us per call, TFLOP/s = 2*M*N*K / time")
    print("%-30s %-6s %10s %10s %9s %9s" % ("layer", "pass", "CT us", "conv us", "CT TF/s", "conv TF/s"))
    for cin, cout, hi, k, s, p, op in CT_SHAPES:
        ho = (hi - 1) * s - 2 * p + k + op
        geom = (n, cout, ho, ho, cin, k, p, s)   # the mirrored convolution: C = out, H = output size, K = in
        flops = 2.0 * n * hi * hi * cin * cout * k * k
        ws, ws_n = ws_for(geom)
        # ConvTranspose2d operands: input x (N,hi,hi,in), weight (in,k,k,out) channels-last, output y, gradients gy / gx / gw
        x, w, y, gy, gx, gw = (dev_rand(n * hi * hi * cin), dev_rand(cin * k * k * cout), m.Array(n * ho * ho * cout),
                               dev_rand(n * ho * ho * cout), m.Array(n * hi * hi * cin), m.Array(cin * k * k * cout))
        # Conv2d(out -> in, k, s, p) operands: input cx (N,ho,ho,out), its output gradient cdy (N,hi,hi,in), cdx, cw, cdw
        cx, cw, cdy, cdx, cdw, cy = (dev_rand(n * ho * ho * cout), dev_rand(cin * k * k * cout), dev_rand(n * hi * hi * cin),
                                     m.Array(n * ho * ho * cout), m.Array(cin * k * k * cout), m.Array(n * hi * hi * cin))
        ct = {"fwd": lambda: m.conv2d_dgrad(x, w, y, *geom, mode, m.DGRAD_EXACT, ws, ws_n, m.WLAYOUT_KRSC),
              "dx": lambda: m.conv2d_fprop(gy, m.LAYOUT_NHWC, w, gx, *geom, mode, ws, ws_n, m.WLAYOUT_KRSC),
              "dw": lambda: m.conv2d_wgrad(gy, m.LAYOUT_NHWC, x, gw, *geom, mode, ws, ws_n, m.WLAYOUT_KRSC)}
        conv = {"fwd": lambda: m.conv2d_dgrad(cdy, cw, cdx, *geom, mode, m.DGRAD_EXACT, ws, ws_n, m.WLAYOUT_KRSC),
                "dx": lambda: m.conv2d_fprop(cx, m.LAYOUT_NHWC, cw, cy, *geom, mode, ws, ws_n, m.WLAYOUT_KRSC),
                "dw": lambda: m.conv2d_wgrad(cx, m.LAYOUT_NHWC, cdy, cdw, *geom, mode, ws, ws_n, m.WLAYOUT_KRSC)}
        name = "%d->%d %d->%d k%d s%d p%d op%d" % (cin, cout, hi, ho, k, s, p, op)
        for pas in ("fwd", "dx", "dw"):
            a, b = [], []
            for _ in range(3):   # alternate the two calls so that both see the same clocks
                a.append(time_it(ct[pas]))
                b.append(time_it(conv[pas]))
            ta, tb = float(np.median(a)), float(np.median(b))
            print("%-30s %-6s %10.1f %10.1f %9.1f %9.1f" % (name, pas, ta, tb, flops / ta / 1e6, flops / tb / 1e6))
            res["conv_transpose"].append({"layer": name, "pass": pas, "ct_us": ta, "conv_us": tb, "ct_tflops": flops / ta / 1e6,
                                          "conv_tflops": flops / tb / 1e6, "ct_runs_us": a, "conv_runs_us": b})
        # the host layer issues exactly one kernel launch for its forward pass (input already channels-last)
        layer = nn.ConvTranspose2d(cin, cout, k, padding=p, stride=s, output_padding=op, bias=False, device="cuda")
        xt = Tensor(backend_api.Btensor(rng.randn(n, cin, hi, hi).astype(np.float32), device=dev).channels_last())
        with tensor.no_grad():
            layer(xt)
            l0 = dev.launch_count()
            layer(xt)
            launches = dev.launch_count() - l0
        print("%-30s host layer forward: %d kernel launch(es)" % (name, launches))
        res.setdefault("layer_fwd_launches", {})[name] = launches
        del x, w, y, gy, gx, gw, cx, cw, cdy, cdx, cdw, cy, ws, layer, xt

    print("\nUpsample: GB/s against the minimum bytes 4 * (1 + s^2) * |x| (read the input once, write the output once)")
    print("%-30s %-9s %-4s %10s %9s" % ("shape", "mode", "pass", "us", "GB/s"))
    for c, h, s in UP_SHAPES:
        nx = n * h * h * c
        x, y, gy, gx = dev_rand(nx), m.Array(nx * s * s), dev_rand(nx * s * s), m.Array(nx)
        nbytes = 4.0 * (1 + s * s) * nx
        for mname, mv in (("nearest", m.UPSAMPLE_NEAREST), ("bilinear", m.UPSAMPLE_BILINEAR)):
            for pas, fn in (("fwd", lambda: m.upsample2d_fwd(x, y, n, h, h, c, s, mv)),
                            ("bwd", lambda: m.upsample2d_bwd(gy, gx, n, h, h, c, s, mv))):
                t = time_it(fn)
                shape = "%dx%dx%dx%d x%d" % (n, c, h, h, s)
                print("%-30s %-9s %-4s %10.1f %9.0f" % (shape, mname, pas, t, nbytes / t / 1e3))
                res["upsample"].append({"shape": shape, "mode": mname, "pass": pas, "us": t, "gbs": nbytes / t / 1e3})
        del x, y, gy, gx

    # the generator's captured training step
    df = workloads.namespace(DeepFlows)
    np.random.seed(0)
    model = workloads.dcgan_generator(df, "cuda")
    opt = df.optim.Adam(model.parameters(), lr=2e-4)
    crit = nn.MSELoss()
    z = Tensor(backend_api.Btensor(rng.randn(n, 64).astype(np.float32), device=dev))
    target = Tensor(backend_api.Btensor(np.tanh(rng.randn(n, 3, 64, 64)).astype(np.float32), device=dev))

    def step_fn():
        loss = crit(model(z), target)
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
    print("\ndcgan_generator training step (batch %d, 64x64x3 output, Adam, captured): %.3f ms/step, %.0f images/s"
          % (n, ms, n / ms * 1e3))
    res["generator"] = {"ms_per_step": ms, "images_per_s": n / ms * 1e3, "steps": args.steps}
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "decoder_bench.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
