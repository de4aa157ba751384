"""Rates of filtered sampling (image_compression.sample / sample_codes) against the compositions a caller would otherwise
write, one JSON line per workload:

  A  2-D model of BASELINE config 2 (4096^2 frame, C = 12), mip 0, Q uniformly random (u, v), bilinear, f16, uint8 out:
     the fused `sample` against torch tap expansion + `decode_points` (fp32 out) + torch blend + the same uint8 rounding;
  B  the 65^3 colour LUT of config 4 from 8-bit codes, trilinear, align_corners: the fused `sample_codes` against a dense
     decode of all 65^3 texels + torch.nn.functional.grid_sample (a measurement: for a model this small the dense route
     may win);
  C  the mip-mapped material stack of config 3 (2048^2, mips 0 .. 11, 9 output channels), f16, uint8 out, Q uniformly
     random (u, v) with a per-query lambda uniform in [0, 8): the fused `sample(lod=tensor)` against the caller's
     composition (torch sort by floor(lambda), scalar `sample` at m and m + 1 per bucket, torch blend, unsort);
  C' the same model at a constant lambda = 1.5: the fused per-query pass against scalar `sample(lod=1.5)` (two passes);
  D  a 3840 x 2160 view of the config-3 texture on a ground plane in perspective, analytic (u, v) and derivatives, wrap
     addressing, through `grad=` (coherent queries, as a renderer issues them), against the same composition.

Timing: CUDA events around each call after warm-up; the two routes of a workload alternate, and a 256 MB write between
timed calls overwrites the L2 (as bench.py does).  The card's name and power limit are printed with the rates.

  python tools/run_sample.py [--steps 10] [--warmup 3] [--queries 16777216] [--workloads ABCD]"""
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


def decoder(dev, cin, seed, cout=3):
    params = I.make_mlp(cin, cout=cout, seed=seed, gain=2.0)
    dec = ic.ColorDecoder(cin, 64, cout).to(dev)
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


def material_stack(dev):
    """Config 3: a 2048^2 mip-mapped model (every pyramid level), 9 output channels."""
    size = 2048
    var2.update(IMAGE_SIZE=size, TF_NO_MIP=False, MAX_MIP_LEVEL=11)
    gen = torch.Generator(device=dev).manual_seed(41)
    fp = [quantized_grid((12, s, s), gen, dev) for s in I.pyramid_sizes(size, False)]
    return fp, decoder(dev, 73, 42, cout=9), gen


def composition(fp, dec, coords, lam, address="clamp"):
    """What a caller writes without a per-query LOD: sort by floor(lambda), two scalar samples per bucket, blend, unsort
    (fp32 out; lambda clamped to [0, 11] as the library clamps it)."""
    lc = torch.nan_to_num(lam, nan=0.0).clamp(0, 11)
    m = torch.floor(lc)
    t = (lc - m).unsqueeze(1)
    order = torch.argsort(m)
    counts = torch.bincount(m.to(torch.int64), minlength=12).tolist()
    out = torch.empty((coords.shape[0], 9), device=coords.device)
    start = 0
    for mip, n in enumerate(counts):
        if n == 0:
            continue
        idx = order[start:start + n]
        start += n
        c = coords[idx].contiguous()
        a = ic.sample(fp, dec, c, mip, address=address, precision="f16")
        if mip < 11:
            b = ic.sample(fp, dec, c, mip + 1, address=address, precision="f16")
            a = (1 - t[idx]) * a + t[idx] * b
        out[idx] = a
    return out


def to_u8(v):
    return torch.floor(v * 255 + 0.5).clamp_(0, 255).to(torch.uint8)


def workload_c(args, dev, flush, info):
    q = args.queries
    fp, dec, gen = material_stack(dev)
    coords = torch.rand((q, 2), generator=gen, device=dev)
    lam = torch.rand(q, generator=gen, device=dev) * 8

    def fused():
        return ic.sample(fp, dec, coords, lam, precision="f16", out_dtype=torch.uint8)

    def composed():
        return to_u8(composition(fp, dec, coords, lam))

    ms_f, ms_c = alternate([fused, composed], args.steps, args.warmup, flush)
    diff = float((ic.sample(fp, dec, coords, lam, precision="f16") - composition(fp, dec, coords, lam)).abs().max())
    print(json.dumps({"workload": "C: config 3 (2048^2, mips 0..11, 9 channels), lambda uniform in [0, 8), f16, uint8 out",
                      "queries": q, "steps": args.steps, "fused_ms": ms_f, "fused_gquery_s": q / ms_f / 1e6,
                      "fused_gtap_s": 8 * q / ms_f / 1e6, "composition_ms": ms_c, "composition_gquery_s": q / ms_c / 1e6,
                      "speedup": ms_c / ms_f, "max_abs_diff_f32": diff, "l2": "overwritten between timed calls", **info}),
          flush=True)
    const = torch.full((q,), 1.5, device=dev)

    def fused_const():
        return ic.sample(fp, dec, coords, const, precision="f16", out_dtype=torch.uint8)

    def scalar():
        return ic.sample(fp, dec, coords, 1.5, precision="f16", out_dtype=torch.uint8)

    ms_f, ms_s = alternate([fused_const, scalar], args.steps, args.warmup, flush)
    diff = float((ic.sample(fp, dec, coords, const, precision="f16") - ic.sample(fp, dec, coords, 1.5, precision="f16")).abs().max())
    print(json.dumps({"workload": "C': config 3, constant lambda = 1.5, f16, uint8 out", "queries": q, "steps": args.steps,
                      "fused_ms": ms_f, "fused_gquery_s": q / ms_f / 1e6, "fused_gtap_s": 8 * q / ms_f / 1e6,
                      "scalar_two_pass_ms": ms_s, "scalar_gquery_s": q / ms_s / 1e6, "speedup": ms_s / ms_f,
                      "max_abs_diff_f32": diff, "l2": "overwritten between timed calls", **info}), flush=True)
    var2.update()


def perspective_plane(width, height, dev):
    """Pixel centres of a ground plane seen from above it: (u, v) = (0.25 sx / sy, 0.25 / sy) with sx in [-1, 1] across the
    screen and sy in (0.02, 1] from the horizon down, and their analytic screen-space derivatives."""
    py, px = torch.meshgrid(torch.arange(height, device=dev, dtype=torch.float32) + 0.5,
                            torch.arange(width, device=dev, dtype=torch.float32) + 0.5, indexing="ij")
    sx = px / width * 2 - 1
    sy = py / height * 0.98 + 0.02
    dsx, dsy = 2.0 / width, 0.98 / height
    u, v = 0.25 * sx / sy, 0.25 / sy
    ddx = torch.stack([0.25 * dsx / sy, torch.zeros_like(sy)], -1)
    ddy = torch.stack([-0.25 * sx / sy ** 2 * dsy, -0.25 / sy ** 2 * dsy], -1)
    flat = lambda t: t.reshape(width * height, -1).contiguous()
    return flat(torch.stack([u, v], -1)), flat(ddx), flat(ddy)


def workload_d(args, dev, flush, info):
    fp, dec, _ = material_stack(dev)
    coords, ddx, ddy = perspective_plane(3840, 2160, dev)
    q = coords.shape[0]
    e0 = 2048.0
    sx, sy = ((ddx * e0) ** 2).sum(1), ((ddy * e0) ** 2).sum(1)
    lam = 0.5 * torch.log2(torch.maximum(sx, sy))

    def fused():
        return ic.sample(fp, dec, coords, grad=(ddx, ddy), address="wrap", precision="f16", out_dtype=torch.uint8)

    def composed():
        return to_u8(composition(fp, dec, coords, lam, address="wrap"))

    ms_f, ms_c = alternate([fused, composed], args.steps, args.warmup, flush)
    diff = float((ic.sample(fp, dec, coords, grad=(ddx, ddy), address="wrap", precision="f16") -
                  composition(fp, dec, coords, lam, address="wrap")).abs().max())
    print(json.dumps({"workload": "D: 3840x2160 perspective ground plane, config-3 texture, grad=, wrap, f16, uint8 out",
                      "queries": q, "lambda_min": float(lam.min()), "lambda_max": float(lam.max()), "steps": args.steps,
                      "fused_ms": ms_f, "fused_gquery_s": q / ms_f / 1e6, "fused_gtap_s": 8 * q / ms_f / 1e6,
                      "composition_ms": ms_c, "composition_gquery_s": q / ms_c / 1e6, "speedup": ms_c / ms_f,
                      "max_abs_diff_f32": diff, "l2": "overwritten between timed calls", **info}), flush=True)
    var2.update()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--queries", type=int, default=1 << 24)
    ap.add_argument("--workloads", default="ABCD")
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
    if "C" in args.workloads:
        workload_c(args, dev, flush, info)
    if "D" in args.workloads:
        workload_d(args, dev, flush, info)
    var2.update()


if __name__ == "__main__":
    main()
