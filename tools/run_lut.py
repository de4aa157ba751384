"""Rates of applying a baked 3-D colour LUT (image_compression.bake_lut_codes + BakedLut.apply) against the routes a caller
has without it, one JSON line per workload.  The model is the 65^3 LUT of BASELINE config 4 from 8-bit codes (the grids and
decoder of tools/run_sample.py workload B).

  A  one 3840 x 2160 uint8 RGB frame (seeded smooth image + noise): fp16-table apply (trilinear, tetrahedral), fp32-table
     apply, `sample_codes` on v / 255 coordinates (today's product route), a dense `decode_codes` + grid_sample + uint8
     rounding (the torch composition), and grid_sample alone on a dense LUT decoded beforehand;
  B  120 frames of 1920 x 1080 (the config-5 clip shape) in one call, 249 M pixels, beyond the L2: Gpixel/s and the share of
     the 6 B/pixel HBM bound (uint8 RGB in and out) at the 6,459.6 GB/s copy rate DESIGN uses;
  C  2^24 uniformly random uint8 pixels: the incoherent worst case for the table gathers;
  D  the bake: dense decode_codes of the 65^3 texels + nic_lut_pack, and the pack alone, in microseconds.

Every workload reports the largest uint8 difference against the fp32-table trilinear arm (trilinear routes) or the fp32-table
tetrahedral arm (tetrahedral routes).  Timing: CUDA events around each call after warm-up; the routes of a workload alternate,
and a 256 MB write between timed calls overwrites the L2.  The card's name and power limit are printed with the rates.

  python tools/run_lut.py [--steps 10] [--warmup 3] [--workloads ABCD]"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from neural_image_compression_v2_b200 import fp_def, var2  # noqa: E402
from neural_image_compression_v2_b200 import image_compression as ic  # noqa: E402
from run_sample import alternate, card, decoder, quantized_grid  # noqa: E402

HBM_COPY_GBS = 6459.6        # DESIGN §4: measured HBM copy rate of the B200


def lut_model(dev):
    """The config-4 model of run_sample.py workload B: (codes, decoder, level table)."""
    var2.update(IMAGE_SIZE=64, IMAGE_DIMENSION=3, COMPRESSION_METHOD=3)
    gen = torch.Generator(device=dev).manual_seed(31)
    fp = [quantized_grid((12, 18, 18, 18), gen, dev), quantized_grid((12, 10, 10, 10), gen, dev)]
    return fp_def.fp_savable(fp, 8), decoder(dev, 127, 32), {0: 0}


def smooth_frames(frames, h, w, seed, dev):
    """[frames, h, w, 3] uint8: a seeded smooth image with noise, shifted from frame to frame (coherent like video)."""
    g = torch.Generator(device=dev).manual_seed(seed)
    low = torch.rand((1, 3, h // 64 + 4, w // 64 + 4), generator=g, device=dev)
    base = torch.nn.functional.interpolate(low, size=(h + 2 * frames, w + 2 * frames), mode="bicubic", align_corners=False)[0]
    out = torch.empty((frames, h, w, 3), dtype=torch.uint8, device=dev)
    for f in range(frames):
        img = base[:, f:f + h, 2 * f:2 * f + w].permute(1, 2, 0) + 0.03 * torch.randn((h, w, 3), generator=g, device=dev)
        out[f] = torch.floor(img.clamp(0, 1) * 255 + 0.5).to(torch.uint8)
    return out


def u8_diff(a, b):
    return int((a.to(torch.int16) - b.to(torch.int16)).abs().max()) if a.numel() else 0


def bakes(codes, dec, table):
    """(fp16-table LUT from the codes, fp32-table LUT of the same model)."""
    lut16 = ic.bake_lut_codes(codes, dec, 8, 0, size=65, precision="f16", level_table=table)
    lut32 = ic.bake_lut(fp_def.fp_load(codes, 8), dec, 0, size=65, precision="f32", level_table=table)
    return lut16, lut32


def workload_a(args, dev, flush, info):
    codes, dec, table = lut_model(dev)
    lut16, lut32 = bakes(codes, dec, table)
    img = smooth_frames(1, 2160, 3840, 51, dev)[0]
    flat = img.view(-1, 3)
    q = flat.shape[0]
    dense_cached = ic.decode_codes(codes, dec, 8, 0, size=65, precision="f16", out_dtype=torch.float32, level_table=table)

    def grid_of(x):
        return (x.to(torch.float32) / 255 * 2 - 1).view(1, q, 1, 1, 3)

    def grid_sample(lut):
        vol = lut.permute(3, 2, 1, 0).unsqueeze(0)                      # [1, C, z, y, x]: grid (x, y, z) indexes (W, H, D)
        v = torch.nn.functional.grid_sample(vol, grid_of(flat), mode="bilinear", padding_mode="border", align_corners=True)
        return torch.floor(v.view(3, q).T * 255 + 0.5).clamp_(0, 255).to(torch.uint8)

    routes = {
        "apply_f16_trilinear": lambda: lut16.apply(img, "trilinear"),
        "apply_f16_tetrahedral": lambda: lut16.apply(img, "tetrahedral"),
        "apply_f32_trilinear": lambda: lut32.apply(img, "trilinear"),
        "sample_codes": lambda: ic.sample_codes(codes, dec, flat.to(torch.float32) / 255, 8, 0, size=65, align_corners=True,
                                                precision="f16", out_dtype=torch.uint8, level_table=table),
        "dense_decode_grid_sample": lambda: grid_sample(ic.decode_codes(codes, dec, 8, 0, size=65, precision="f16",
                                                                        out_dtype=torch.float32, level_table=table)),
        "grid_sample_cached_dense": lambda: grid_sample(dense_cached),
    }
    ms = dict(zip(routes, alternate(list(routes.values()), args.steps, args.warmup, flush)))
    ref_tri = lut32.apply(img, "trilinear").view(-1, 3)
    ref_tet = lut32.apply(img, "tetrahedral").view(-1, 3)
    diff = {k: u8_diff(r().reshape(-1, 3), ref_tet if "tetrahedral" in k else ref_tri) for k, r in routes.items()}
    rates = {k: q / v / 1e6 for k, v in ms.items()}
    best_baked = min(ms["apply_f16_trilinear"], ms["apply_f16_tetrahedral"])
    print(json.dumps({"workload": "A: one 3840x2160 uint8 RGB frame, config-4 65^3 LUT from 8-bit codes, uint8 out",
                      "pixels": q, "steps": args.steps, "ms": ms, "gpixel_s": rates, "u8_max_diff_vs_f32_table": diff,
                      "speedup_f16_trilinear_vs_dense_decode_grid_sample":
                          ms["dense_decode_grid_sample"] / ms["apply_f16_trilinear"],
                      "baked_apply_beats_dense_decode_grid_sample": best_baked < ms["dense_decode_grid_sample"],
                      "l2": "overwritten between timed calls", **info}), flush=True)
    var2.update()


def workload_b(args, dev, flush, info):
    codes, dec, table = lut_model(dev)
    lut16, lut32 = bakes(codes, dec, table)
    clip = smooth_frames(120, 1080, 1920, 52, dev)
    q = clip.numel() // 3
    out = torch.empty_like(clip)
    routes = {"apply_f16_trilinear": lambda: lut16.apply(clip, "trilinear", out=out),
              "apply_f16_tetrahedral": lambda: lut16.apply(clip, "tetrahedral", out=out)}
    ms = dict(zip(routes, alternate(list(routes.values()), args.steps, args.warmup, flush)))
    diff = {}
    for k, interp in (("apply_f16_trilinear", "trilinear"), ("apply_f16_tetrahedral", "tetrahedral")):
        diff[k] = u8_diff(lut16.apply(clip, interp), lut32.apply(clip, interp))
    bound_ms = 6.0 * q / (HBM_COPY_GBS * 1e9) * 1e3
    print(json.dumps({"workload": "B: 120 frames of 1920x1080 uint8 RGB in one call (config-5 clip shape), 65^3 LUT, uint8 out",
                      "pixels": q, "steps": args.steps, "ms": ms, "gpixel_s": {k: q / v / 1e6 for k, v in ms.items()},
                      "hbm_bound_ms_6B_per_pixel": bound_ms, "hbm_bound_gbs": HBM_COPY_GBS,
                      "fraction_of_hbm_bound": {k: bound_ms / v for k, v in ms.items()},
                      "u8_max_diff_vs_f32_table": diff, "l2": "working set 1.5 GB, beyond the L2", **info}), flush=True)
    var2.update()


def workload_c(args, dev, flush, info):
    codes, dec, table = lut_model(dev)
    lut16, lut32 = bakes(codes, dec, table)
    gen = torch.Generator(device=dev).manual_seed(53)
    px = torch.randint(0, 256, (1 << 24, 3), generator=gen, device=dev, dtype=torch.int32).to(torch.uint8)
    q = px.shape[0]
    routes = {"apply_f16_trilinear": lambda: lut16.apply(px, "trilinear"),
              "apply_f16_tetrahedral": lambda: lut16.apply(px, "tetrahedral"),
              "apply_f32_trilinear": lambda: lut32.apply(px, "trilinear")}
    ms = dict(zip(routes, alternate(list(routes.values()), args.steps, args.warmup, flush)))
    diff = {k: u8_diff(r(), lut32.apply(px, "tetrahedral" if "tetrahedral" in k else "trilinear")) for k, r in routes.items()}
    print(json.dumps({"workload": "C: 2^24 uniformly random uint8 pixels, 65^3 LUT, uint8 out", "pixels": q,
                      "steps": args.steps, "ms": ms, "gpixel_s": {k: q / v / 1e6 for k, v in ms.items()},
                      "u8_max_diff_vs_f32_table": diff, "l2": "overwritten between timed calls", **info}), flush=True)
    var2.update()


def workload_d(args, dev, flush, info):
    codes, dec, table = lut_model(dev)
    dense = ic.decode_codes(codes, dec, 8, 0, size=65, precision="f16", out_dtype=torch.float32, level_table=table)
    routes = {"bake_lut_codes_f16": lambda: ic.bake_lut_codes(codes, dec, 8, 0, size=65, precision="f16", level_table=table),
              "pack_only_f16": lambda: ic.BakedLut.from_table(dense, torch.float16)}
    ms = dict(zip(routes, alternate(list(routes.values()), args.steps, args.warmup, flush)))
    print(json.dumps({"workload": "D: bake of the config-4 65^3 LUT from 8-bit codes (decode_codes + nic_lut_pack)",
                      "texels": 65 ** 3, "steps": args.steps, "us": {k: v * 1e3 for k, v in ms.items()},
                      "l2": "overwritten between timed calls", **info}), flush=True)
    var2.update()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workloads", default="ABCD")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("run_lut.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda:0")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)        # > the 126 MB L2
    info = card()
    for w, fn in (("A", workload_a), ("B", workload_b), ("C", workload_c), ("D", workload_d)):
        if w in args.workloads:
            fn(args, dev, flush, info)
    var2.update()


if __name__ == "__main__":
    main()
