"""Rates of decoding a whole mip chain (image_compression.decode_mips / decode_mips_codes) against the Python loop a caller
would otherwise write (one `decode` / `decode_codes` per mip), one JSON line per workload:

  A  the config-2 shape with a mip pyramid: a 4096^2 RGB model (C = 12, every pyramid level), mips 0 .. 12, f16, uint8 out;
  B  the config-3 material stack: 2048^2, 9 output channels, mips 0 .. 11, bf16, uint8 out;
  C  a 256^3 method-3 volume, mips 0 .. 8, f16, uint8 out;
  A' A from 8-bit codes (decode_mips_codes against a loop of decode_codes).

Both routes rebuild their tables on every call (no DecodeSession).  Per route: ms per chain, Gtexel/s over the whole chain,
kernel launches per chain (nic_launch_count), the host time to enqueue one chain without a synchronise, and the largest
8-bit difference of decode_mips from the loop, at mip 0 and over mips >= 1.

Timing: CUDA events around each call after warm-up; the two routes of a workload alternate, and a 256 MB write between
timed calls overwrites the L2 (as run_sample.py and bench.py do).  The card's name and power limit are printed with the rates.

  python tools/run_mips.py [--steps 10] [--warmup 3] [--workloads ABCa]     (a = A')"""
import argparse
import json
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from run_sample import I, alternate, card, decoder, fp_def, ic, quantized_grid, var2  # noqa: E402
import neural_image_compression_v2_b200 as nic  # noqa: E402


def enqueue_ms(route, reps=5):
    """Host time of one call that returns without a synchronise (the device then drains before the next one)."""
    total = 0.0
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        route()
        total += time.perf_counter() - t0
    torch.cuda.synchronize()
    return total / reps * 1e3


def launches(route, dev):
    before = nic.launch_count(dev)
    route()
    return nic.launch_count(dev) - before


def measure(name, args, dev, flush, info, chain, loop, last):
    ms_c, ms_l = alternate([chain, loop], args.steps, args.warmup, flush)
    a, b = chain(), loop()
    diff = [int((x.to(torch.int16) - y.to(torch.int16)).abs().max()) for x, y in zip(a, b)]
    texels = sum(x.numel() // x.shape[-1] for x in a)
    print(json.dumps({"workload": name, "mips": last + 1, "texels": texels, "steps": args.steps,
                      "decode_mips_ms": ms_c, "decode_mips_gtexel_s": texels / ms_c / 1e6,
                      "loop_ms": ms_l, "loop_gtexel_s": texels / ms_l / 1e6, "speedup": ms_l / ms_c,
                      "decode_mips_launches": launches(chain, dev), "loop_launches": launches(loop, dev),
                      "decode_mips_enqueue_ms": enqueue_ms(chain), "loop_enqueue_ms": enqueue_ms(loop),
                      "u8_max_diff_mip0": diff[0], "u8_max_diff_mips_1_up": max(diff[1:]),
                      "l2": "overwritten between timed calls", **info}), flush=True)


def routes(fp, dec, last, precision, codes=None, bits=8):
    """(decode_mips, the per-mip loop) of mips 0 .. last, uint8 out."""
    if codes is None:
        return (lambda: ic.decode_mips(fp, dec, precision=precision, out_dtype=torch.uint8),
                lambda: [ic.decode(fp, dec, i, precision=precision, out_dtype=torch.uint8) for i in range(last + 1)])
    return (lambda: ic.decode_mips_codes(codes, dec, bits, precision=precision, out_dtype=torch.uint8),
            lambda: [ic.decode_codes(codes, dec, bits, i, precision=precision, out_dtype=torch.uint8) for i in range(last + 1)])


def pyramid(size, dim, seed, dev):
    gen = torch.Generator(device=dev).manual_seed(seed)
    return [quantized_grid((12,) + (s,) * dim, gen, dev) for s in I.pyramid_sizes(size, False)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workloads", default="ABCa")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("run_mips.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda:0")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)        # > the 126 MB L2
    info = card()
    if "A" in args.workloads or "a" in args.workloads:
        var2.update(IMAGE_SIZE=4096, TF_NO_MIP=False, MAX_MIP_LEVEL=12)
        fp, dec = pyramid(4096, 2, 51, dev), decoder(dev, 73, 52)
        if "A" in args.workloads:
            measure("A: config-2 shape, 4096^2 RGB C=12, mips 0..12, f16, uint8 out", args, dev, flush, info,
                    *routes(fp, dec, 12, "f16"), 12)
        if "a" in args.workloads:
            codes = fp_def.fp_savable(fp, 8)
            measure("A': A from 8-bit codes", args, dev, flush, info, *routes(None, dec, 12, "f16", codes, 8), 12)
            del codes
        del fp
    if "B" in args.workloads:
        var2.update(IMAGE_SIZE=2048, TF_NO_MIP=False, MAX_MIP_LEVEL=11)
        fp, dec = pyramid(2048, 2, 41, dev), decoder(dev, 73, 42, cout=9)
        measure("B: config-3 material stack, 2048^2 x 9 channels, mips 0..11, bf16, uint8 out", args, dev, flush, info,
                *routes(fp, dec, 11, "bf16"), 11)
        del fp
    if "C" in args.workloads:
        var2.update(IMAGE_SIZE=256, IMAGE_DIMENSION=3, COMPRESSION_METHOD=3, TF_NO_MIP=False, MAX_MIP_LEVEL=8)
        fp, dec = pyramid(256, 3, 61, dev), decoder(dev, 127, 62)
        measure("C: 256^3 method-3 volume, mips 0..8, f16, uint8 out", args, dev, flush, info, *routes(fp, dec, 8, "f16"), 8)
        del fp
    var2.update()


if __name__ == "__main__":
    main()
