#!/usr/bin/env python
"""Per-op microbenchmark on one B200: every conv (fprop / dgrad / wgrad) and BatchNorm (fwd / bwd) shape of the
ResNet-18/CIFAR step at batch 256 (and optional 224x224 VGG layers), timed with CUDA events on the library's
compute stream, L2 flushed between iterations, against the roofline max(t_HBM, t_TC) of SURVEY 8d.

    python scripts/opbench.py [--batch 256] [--iters 20] [--big] [--mode tf32] [--json out.json]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import deepflows_b200  # noqa: E402,F401
import bench  # noqa: E402


def event_timer(m, iters, flush=None, graph=False):
    """time_it(fn) -> microseconds per call of fn on the library's compute stream, CUDA events around each of `iters`
    calls after 3 warm-up calls, the L2 overwritten before each (`flush`: a device Array larger than the L2, or None).
    graph=True: 20 back-to-back calls replayed from one CUDA graph instead (no host launch cost, warm L2)."""
    def time_it(fn):
        for _ in range(3):
            fn()
        if graph:
            reps = 20
            m.graph_begin_capture()
            for _ in range(reps):
                fn()
            g = m.graph_end_capture()
            for _ in range(2):
                m.graph_launch(g)
            e0, e1 = m.event_create(), m.event_create()
            m.event_record(e0)
            for _ in range(5):
                m.graph_launch(g)
            m.event_record(e1)
            m.event_synchronize(e1)
            us = m.event_elapsed_ms(e0, e1) / (5 * reps) * 1e3
            m.event_destroy(e0)
            m.event_destroy(e1)
            m.graph_destroy(g)
            return us
        tot = 0.0
        e0, e1 = m.event_create(), m.event_create()
        for _ in range(iters):
            if flush is not None:
                m.fill(flush, 0.0)
            m.event_record(e0)
            fn()
            m.event_record(e1)
            m.event_synchronize(e1)
            tot += m.event_elapsed_ms(e0, e1)
        m.event_destroy(e0)
        m.event_destroy(e1)
        return tot / iters * 1e3  # us

    return time_it


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--big", action="store_true", help="add 224x224 VGG-16 layers (tensor-pipe bound)")
    ap.add_argument("--mode", default="tf32")
    ap.add_argument("--json", default=None)
    ap.add_argument("--no-flush", action="store_true")
    ap.add_argument("--graph", action="store_true",
                    help="time each op as 20 back-to-back calls replayed from one CUDA graph (no host launch cost, "
                         "warm L2): what the op costs inside the captured training step")
    args = ap.parse_args()
    from DeepFlows import backend_api
    dev = backend_api.cuda()
    m = dev.mod
    mode = {"fp32": m.MODE_FP32, "tf32": m.MODE_TF32, "bf16": m.MODE_BF16}[args.mode]
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
    hbm = peaks.get("hbm_gbs", 6650.0) * 1e9
    tc = peaks.get("bf16_tflops", 1590.0) * 1e12 / 2  # TF32 dense = half the bf16 rate
    flush = m.Array(64 << 20)  # 256 MB > 126 MB L2
    rng = np.random.RandomState(0)

    time_it = event_timer(m, args.iters, None if args.no_flush else flush, args.graph)

    def dev_rand(n):
        a = m.Array(n)
        m.from_numpy(rng.randn(n).astype(np.float32), a)
        return a

    rows = []
    layers = bench.conv_layers(args.batch)
    if args.big:
        b = 32
        layers += [("vgg.c1_2", b, 64, 224, 224, 64, 3, 1, 1, 1), ("vgg.c2_2", b, 128, 112, 112, 128, 3, 1, 1, 1),
                   ("vgg.c3_2", b, 256, 56, 56, 256, 3, 1, 1, 1), ("vgg.c4_2", b, 512, 28, 28, 512, 3, 1, 1, 1)]
    seen = {}
    print("%-14s %-28s %9s %9s %7s  %9s %7s  %9s %7s" % ("layer", "N,C,H,W,K,R,p,s", "roof us", "fprop us", "frac", "dgrad us", "frac", "wgrad us", "frac"))
    tot = {"roof": 0.0, "fprop": 0.0, "dgrad": 0.0, "wgrad": 0.0}
    for (name, n, c, h, w, k, r, p, s, _cnt) in layers:
        geom = (n, c, h, w, k, r, p, s)
        oh, ow = (h + 2 * p - r) // s + 1, (w + 2 * p - r) // s + 1
        flops = 2.0 * n * oh * ow * k * c * r * r
        bytes_min = 4.0 * (n * c * h * w + k * c * r * r + n * oh * ow * k)
        roof = max(flops / tc, bytes_min / hbm) * 1e6
        if geom not in seen:
            x, wt, y = dev_rand(n * c * h * w), dev_rand(k * c * r * r), m.Array(n * oh * ow * k)
            gy, dx, dw = dev_rand(n * oh * ow * k), m.Array(n * c * h * w), m.Array(k * c * r * r)
            tf = time_it(lambda: m.conv2d_fprop(x, m.LAYOUT_NHWC, wt, y, n, c, h, w, k, r, p, s, mode, None, 0))
            td = time_it(lambda: m.conv2d_dgrad(gy, wt, dx, n, c, h, w, k, r, p, s, mode, m.DGRAD_EXACT, None, 0))
            tw = time_it(lambda: m.conv2d_wgrad(x, m.LAYOUT_NHWC, gy, dw, n, c, h, w, k, r, p, s, mode, None, 0))
            seen[geom] = (tf, td, tw)
            del x, wt, y, gy, dx, dw
        else:
            tf, td, tw = seen[geom]
        print("%-14s %-28s %9.1f %9.1f %7.3f  %9.1f %7.3f  %9.1f %7.3f" % (name, ",".join(map(str, geom)), roof, tf, roof / tf, td, roof / td, tw, roof / tw))
        rows.append({"layer": name, "geom": geom, "roof_us": roof, "fprop_us": tf, "dgrad_us": td, "wgrad_us": tw, "gflop": flops / 1e9,
                     "min_mb": bytes_min / 1e6})
        if not name.startswith("vgg"):
            tot["roof"] += roof; tot["fprop"] += tf; tot["dgrad"] += td if name != "stem" else 0.0; tot["wgrad"] += tw
    print("conv totals per step (us): roofline(one pass) %.1f  fprop %.1f  dgrad %.1f  wgrad %.1f" % (tot["roof"], tot["fprop"], tot["dgrad"], tot["wgrad"]))

    print("\n%-22s %9s %9s %7s %9s %9s %7s" % ("batchnorm rows x C", "fwd roof", "fwd us", "GB/s", "bwd roof", "bwd us", "GB/s"))
    bn_shapes = []
    for (name, n, c, h, w, k, r, p, s, _cnt) in bench.conv_layers(args.batch):
        oh = (h + 2 * p - r) // s + 1
        bn_shapes.append((n * oh * oh, k))
    bt = {"f": 0.0, "b": 0.0, "fr": 0.0, "br": 0.0}
    cache = {}
    for rws, c in bn_shapes:
        if (rws, c) not in cache:
            x, gy, y, dx = dev_rand(rws * c), dev_rand(rws * c), m.Array(rws * c), m.Array(rws * c)
            g, b_, mean, inv, rm, rv, dg, db = [dev_rand(c) for _ in range(8)]
            m.fill(rv, 1.0)
            tfw = time_it(lambda: m.bn_fwd_train(x, g, b_, y, mean, inv, rm, rv, 0.1, 1e-5, rws, c))
            tbw = time_it(lambda: m.bn_bwd(x, gy, g, mean, inv, dx, dg, db, rws, c))
            cache[(rws, c)] = (tfw, tbw)
            del x, gy, y, dx
        tfw, tbw = cache[(rws, c)]
        fb, bb = 12.0 * rws * c, 20.0 * rws * c
        print("%-22s %9.1f %9.1f %7.0f %9.1f %9.1f %7.0f" % ("%d x %d" % (rws, c), fb / hbm * 1e6, tfw, fb / tfw / 1e3, bb / hbm * 1e6, tbw, bb / tbw / 1e3))
        bt["f"] += tfw; bt["b"] += tbw; bt["fr"] += fb / hbm * 1e6; bt["br"] += bb / hbm * 1e6
        rows.append({"bn": (rws, c), "fwd_us": tfw, "bwd_us": tbw, "fwd_gbs": fb / tfw / 1e3, "bwd_gbs": bb / tbw / 1e3})
    print("batchnorm totals per step (us): fwd %.1f (roofline %.1f)  bwd %.1f (roofline %.1f)" % (bt["f"], bt["fr"], bt["b"], bt["br"]))
    if args.json:
        json.dump(rows, open(args.json, "w"), indent=1)


if __name__ == "__main__":
    main()
