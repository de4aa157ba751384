"""Rates of filtered sampling (image_compression.sample / sample_codes) against the compositions a caller would otherwise
write, one JSON line per workload:

  A  2-D model of BASELINE config 2 (4096^2 frame, C = 12), mip 0, Q uniformly random (u, v), bilinear, f16, uint8 out:
     the fused `sample` against torch tap expansion + `decode_points` (fp32 out) + torch blend + the same uint8 rounding;
  B  the 65^3 colour LUT of config 4 from 8-bit codes, trilinear, align_corners: the fused `sample_codes` against a dense
     decode of all 65^3 texels + torch.nn.functional.grid_sample (a measurement: for a model this small the dense route
     may win).

Timing: CUDA events around each call after warm-up; the two routes of a workload alternate, and a 256 MB write between
timed calls overwrites the L2 (as bench.py does).  The card's name and power limit are printed with the rates.

  python tools/run_sample.py [--steps 10] [--warmup 3] [--queries 16777216] [--workloads AB]"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import inputs as I  # noqa: E402
from neural_image_compression_v2_b200 import fp_def, var2  # noqa: E402
from neural_image_compression_v2_b200 import image_compression as ic  # noqa: E402


def card():
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = None
    return {"device": torch.cuda.get_device_name(0), "power_limit": limit}


def decoder(dev, cin, seed):
    params = I.make_mlp(cin, seed=seed, gain=2.0)
    dec = ic.ColorDecoder(cin, 64, 3).to(dev)
    with torch.no_grad():
        for p, v in zip(dec.parameters_list(), params):
            p.copy_(torch.tensor(v))
    return dec


def quantized_grid(shape, gen, dev):
    lo, hi = I.q_range(8)
    g = torch.rand(shape, generator=gen, device=dev) * (hi - lo) + lo
    return (torch.floor(g * 255 + 0.5) / 255).contiguous()


def alternate(routes, steps, warmup, flush):
    """ms per call of each route; the routes are called in turn, each call between its own event pair."""
    for _ in range(warmup):
        for r in routes:
            r()
    ev = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)] for _ in routes]
    for i in range(steps):
        for r, e in zip(routes, ev):
            flush.zero_()
            e[i][0].record()
            r()
            e[i][1].record()
    torch.cuda.synchronize()
    return [sum(s.elapsed_time(t) for s, t in e) / steps for e in ev]


def bilinear_taps(coords, size):
    """The tap rule of nic.h (align_corners = False, clamp) in torch: int64 taps [Q * 4, 2] (x slowest) and weights [Q, 4]."""
    p = coords * size - 0.5
    p = torch.clamp(p, -2.0 ** 24, 2.0 ** 24)
    i0 = torch.floor(p)
    f = p - i0
    i0 = i0.to(torch.int64)
    ix = torch.stack([i0[:, 0], i0[:, 0], i0[:, 0] + 1, i0[:, 0] + 1], 1).clamp_(0, size - 1)
    iy = torch.stack([i0[:, 1], i0[:, 1] + 1, i0[:, 1], i0[:, 1] + 1], 1).clamp_(0, size - 1)
    wx, wy = torch.stack([1 - f[:, 0], f[:, 0]], 1), torch.stack([1 - f[:, 1], f[:, 1]], 1)
    w = torch.stack([wx[:, 0] * wy[:, 0], wx[:, 0] * wy[:, 1], wx[:, 1] * wy[:, 0], wx[:, 1] * wy[:, 1]], 1)
    return torch.stack([ix, iy], 2).reshape(-1, 2), w


def workload_a(args, dev, flush, info):
    size, q = 4096, args.queries
    var2.update(IMAGE_SIZE=size)
    gen = torch.Generator(device=dev).manual_seed(21)
    fp = [quantized_grid((12, size // 4 + 1, size // 4 + 1), gen, dev), quantized_grid((12, size // 8 + 1, size // 8 + 1), gen, dev)]
    dec = decoder(dev, 73, 22)
    coords = torch.rand((q, 2), generator=gen, device=dev)

    def fused():
        return ic.sample(fp, dec, coords, 0, precision="f16", out_dtype=torch.uint8)

    def unfused(quantize=True):
        taps, w = bilinear_taps(coords, size)
        vals = ic.decode_points(fp, dec, taps, 0, precision="f16", out_dtype=torch.float32).view(q, 4, -1)
        v = (w.unsqueeze(2) * vals).sum(1)
        return torch.floor(v * 255 + 0.5).clamp_(0, 255).to(torch.uint8) if quantize else v

    ms_f, ms_u = alternate([fused, unfused], args.steps, args.warmup, flush)
    a = ic.sample(fp, dec, coords, 0, precision="f16", out_dtype=torch.float32)
    b = unfused(quantize=False)
    diff = float((a - b).abs().max())
    u8 = (fused().to(torch.int32) - unfused().to(torch.int32)).abs()
    print(json.dumps({"workload": "A: 2-D 4096^2 C=12 mip 0, bilinear, f16, uint8 out", "queries": q, "steps": args.steps,
                      "fused_ms": ms_f, "fused_gquery_s": q / ms_f / 1e6, "fused_gtap_s": 4 * q / ms_f / 1e6,
                      "unfused_ms": ms_u, "unfused_gquery_s": q / ms_u / 1e6, "speedup": ms_u / ms_f,
                      "max_abs_diff_f32": diff, "u8_max_diff": int(u8.max()), "l2": "overwritten between timed calls",
                      **info}), flush=True)
    del fp, coords, a, b


def workload_b(args, dev, flush, info):
    q = args.queries
    var2.update(IMAGE_SIZE=64, IMAGE_DIMENSION=3, COMPRESSION_METHOD=3)
    gen = torch.Generator(device=dev).manual_seed(31)
    fp = [quantized_grid((12, 18, 18, 18), gen, dev), quantized_grid((12, 10, 10, 10), gen, dev)]
    codes = fp_def.fp_savable(fp, 8)
    dec = decoder(dev, 127, 32)
    table = {0: 0}
    coords = torch.rand((q, 3), generator=gen, device=dev)
    grid = (coords * 2 - 1).view(1, q, 1, 1, 3)

    def fused():
        return ic.sample_codes(codes, dec, coords, 8, 0, size=65, align_corners=True, precision="f16", level_table=table)

    def dense():
        lut = ic.decode_codes(codes, dec, 8, 0, size=65, precision="f16", out_dtype=torch.float32, level_table=table)
        vol = lut.permute(3, 2, 1, 0).unsqueeze(0)                      # [1, C, z, y, x]: grid (x, y, z) indexes (W, H, D)
        return torch.nn.functional.grid_sample(vol, grid, mode="bilinear", padding_mode="border",
                                               align_corners=True).view(3, q).T

    ms_f, ms_d = alternate([fused, dense], args.steps, args.warmup, flush)
    diff = float((fused() - dense()).abs().max())
    print(json.dumps({"workload": "B: 65^3 LUT (config 4) from 8-bit codes, trilinear, align_corners, f16, f32 out",
                      "queries": q, "steps": args.steps, "fused_ms": ms_f, "fused_gquery_s": q / ms_f / 1e6,
                      "fused_gtap_s": 8 * q / ms_f / 1e6, "dense_grid_sample_ms": ms_d, "dense_gquery_s": q / ms_d / 1e6,
                      "faster": "fused" if ms_f < ms_d else "dense + grid_sample", "ratio": max(ms_f, ms_d) / min(ms_f, ms_d),
                      "max_abs_diff": diff, "l2": "overwritten between timed calls", **info}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--queries", type=int, default=1 << 24)
    ap.add_argument("--workloads", default="AB")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("run_sample.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda:0")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)        # > the 126 MB L2
    info = card()
    if "A" in args.workloads:
        workload_a(args, dev, flush, info)
    if "B" in args.workloads:
        workload_b(args, dev, flush, info)
    var2.update()


if __name__ == "__main__":
    main()
