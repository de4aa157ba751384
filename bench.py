#!/usr/bin/env python
"""bench.py — benchmarks of the decode / training hot path on B200 (DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--prec f16|bf16|f32]
                    [--workload decode_4096|decode_4096_strong|train_2048_mips|lut_65|video_1080p120] [--dump-outputs DIR]

Prints ONE JSON line.  The default workload is BASELINE.json configs[1]: full-frame decode of a 4096x4096 RGB texture on
the tensor-core path, one frame per GPU per step ("weak": frames are independent).  `value` = decoded Gtexel/s over all
ranks with grids and decoder resident in HBM; `e2e` = the same metric through the public API with HOST buffers (pinned H2D
of the compressed grids + decoder, decode, D2H of the 8-bit frame inside the timed region), next to the concurrent N-rank
PCIe floor of the same copies.  `--impl reference` times the CPU port of the reference's algorithm (oracle/) on the host
cores, one whole frame per step.  The other workloads are BASELINE configs 3 / 4 / 5 at their named shapes and the
strong-scaling form of config 2 (one frame tiled over N GPUs); each prints its own line.

`--steps K` is the number of timed steps of every workload and of each of its timed legs.  `--dump-outputs DIR` is
accepted for decode_4096 only: after the timed steps it writes a fixed, seeded sample of the last step's frame to
DIR/frame.npy.  With --gpus N > 1 that is rank 0's frame; every rank decodes its own seeded model.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))

SIZE = 4096                      # BASELINE.json configs[1]
FLOP_2D = 2 * (73 * 64 + 64 * 64 + 64 * 3)             # 17,920 per texel (SURVEY.md §8(d))
FLOP_M3 = 2 * (127 * 64 + 64 * 64 + 64 * 3)            # 24,832 (3-D method 3)
METRIC, UNIT = "decoded Gtexel/s (4096x4096 RGB full-frame decode)", "Gtexel/s"
CPU_TILE = 1024                  # decode_image's own tile size for large frames (image_compression.py:310-312)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops", 1590.0), d.get("hbm_gbs", 6650.0), "measured"
    return 1590.0, 6650.0, "fallback"


def recorded_profile(kernel):
    """Numbers of the committed ncu capture of `kernel` (profiles/CURRENT.json names the summary file): they are RECORDED
    values of that capture, reported next to — never instead of — the timings measured in this run."""
    try:
        cur = json.load(open(os.path.join(ROOT, "profiles", "CURRENT.json")))[kernel]
        txt = open(os.path.join(ROOT, cur["metrics"])).read()

        def num(name):
            m = re.search(re.escape(name) + r" = ([0-9.]+) (\S+)", txt)
            if not m:
                return None
            v = float(m.group(1))
            return v * {"Mbyte": 1e6, "Kbyte": 1e3, "Gbyte": 1e9, "byte": 1.0}.get(m.group(2), 1.0)

        rd, wr = num("dram__bytes_read.sum"), num("dram__bytes_write.sum")
        return {"source": cur["metrics"], "commit": cur.get("commit"),
                "traffic_bytes": (rd + wr) if rd is not None and wr is not None else None,
                "xu_pct_busy": num("sm__inst_executed_pipe_xu.avg.pct_of_peak_sustained_active"),
                "tensor_pct_active": num("sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active"),
                "issue_pct_active": num("smsp__issue_active.avg.pct_of_peak_sustained_active"),
                "duration_us_under_ncu": num("gpu__time_duration.sum")}
    except Exception as e:      # a missing summary must not take the benchmark down
        return {"source": None, "error": str(e), "traffic_bytes": None}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(index), "-lms", "50"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def synthetic_model(seed=0):
    import inputs as I
    grids = I.make_grids(SIZE, 2, seed=seed, no_mip=True, quantized=True)      # [12,1025,1025], [12,513,513]
    params = I.make_mlp(73, seed=seed + 1, gain=2.0)
    return grids, params


def decode_config():
    """The workload description shared by both arms (`--impl ours` and `--impl reference` print the same dict)."""
    return {"workload": "decode_4096x4096_rgb", "frame": "one 4096x4096 RGB frame per GPU per step (16.8 Mtexel)",
            "grids": "[12,1025,1025]+[12,513,513] 8-bit", "decoder": "73-64-64-3", "output": "uint8"}


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_setup(threads):
    import torch
    from oracle import nic_oracle as O
    from oracle import nic_oracle_torch as OT
    torch.set_num_threads(threads)
    grids, params = synthetic_model()
    fp = [torch.tensor(g) for g in grids]
    dec = OT.make_decoder(params)
    table = O.create_pyramid_mip_levels(SIZE, SIZE // 4)
    return OT, fp, dec, table


def cpu_decode_tiles(ctx, tiles, first=0, keep=None):
    """Decodes `tiles` 1024x1024 tiles of the 4096^2 frame with the torch-CPU port of the reference path
    (oracle/nic_oracle_torch.py: the reference's own op sequence incl. the 8-bit output quantiser).  Returns
    (texels, seconds); `keep` (a dict) collects tile index -> uint8 [1024, 1024, 3]."""
    import torch
    OT, fp, dec, table = ctx
    n = SIZE // CPU_TILE
    t0 = time.perf_counter()
    for i in range(first, first + tiles):
        x, y = (i % (n * n)) % n, (i % (n * n)) // n
        with torch.no_grad():
            out = OT.decode_block(fp, dec, CPU_TILE, 0, table, 1, origin=(CPU_TILE * x, CPU_TILE * y))
            u8 = torch.floor(out * 255 + 0.5).to(torch.uint8)
        if keep is not None and (i % (n * n)) not in keep:
            keep[i % (n * n)] = u8.reshape(CPU_TILE, CPU_TILE, 3).numpy()
    return tiles * CPU_TILE * CPU_TILE, time.perf_counter() - t0


def cpu_train_rate(threads, steps=2):
    """Msamples/s of the torch-CPU port of train_models' body at config 1 (8 crops of 256^2 on a 512^2 image)."""
    import torch
    import inputs as I
    from oracle import nic_oracle as O
    from oracle import nic_oracle_torch as OT
    torch.set_num_threads(threads)
    size = 512
    table = O.create_pyramid_mip_levels(size, size // 4)
    tr = OT.Trainer(I.make_grids(size, 2, seed=3, no_mip=True), OT.make_decoder(I.make_mlp(73, seed=4)), 1000, 8, 1, table)
    img = torch.tensor(I.make_image(size, 2, seed=5))
    g = torch.Generator().manual_seed(6)
    dt = 0.0
    for s in range(steps + 1):
        coord = torch.randint(0, size - 256 + 1, (8, 2), generator=g)
        tg = torch.stack([img[:, c[0]:c[0] + 256, c[1]:c[1] + 256].reshape(3, -1).T for c in coord.tolist()])
        t0 = time.perf_counter()
        tr.step(coord, tg, 0)
        if s > 0:
            dt += time.perf_counter() - t0
    return steps * 8 * 256 * 256 / dt / 1e6


def run_reference(args):
    """The reference arm: the reference's own CPU op sequence (oracle port, kind "port": the reference is a Python script
    directory that cannot travel to the GPU box) on all host threads, ONE WHOLE 4096^2 FRAME (16 tiles of 1024^2, the
    reference's own tiling) per step, same config / steps / warm-up as the GPU arm."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload != "decode_4096":
        print(json.dumps({"impl": "reference", "unavailable": f"the reference arm covers the headline workload (decode_4096); "
                                                              f"{args.workload} reports its own cpu_baseline"}))
        return
    threads = os.cpu_count() or 1
    ctx = cpu_setup(threads)
    tiles = (SIZE // CPU_TILE) ** 2
    for w in range(args.warmup):
        cpu_decode_tiles(ctx, tiles)
    done, tot_t = 0, 0.0
    for k in range(args.steps):
        d, dt = cpu_decode_tiles(ctx, tiles)
        done += d
        tot_t += dt
    v = done / tot_t / 1e9
    sample = f"the whole frame: {tiles} tiles of {CPU_TILE}x{CPU_TILE} texels per step"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": decode_config(),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": sample + "; torch-CPU port of the reference op sequence (oracle/nic_oracle_torch.py)"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


# ------------------------------------------------------------------------------------------------ GPU arm: helpers
class Env:
    """Process / device set-up shared by the GPU workloads."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        # stdout carries the ONE JSON line and nothing else: libraries that print to fd 1 (NCCL's banner) go to stderr
        self.real_stdout = os.dup(1)
        os.dup2(2, 1)
        self.numa = bind_to_gpu_numa_node(self.local) if self.world > 1 else None
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, ms):
        t = self.torch.tensor([ms], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def emit(self, line):
        if self.rank == 0:
            sys.stdout.flush()
            os.dup2(self.real_stdout, 1)
            print(json.dumps(line), flush=True)
            os.dup2(2, 1)

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def bind_to_gpu_numa_node(local):
    """Pins this rank (and therefore its first-touch pinned host buffers) to the CPUs of the NUMA node its GPU hangs
    off, so the e2e host<->device copies of different ranks do not all cross the socket interconnect."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(local)],
                             capture_output=True, text=True).stdout.strip()
        bus = out[-12:] if out else None              # 00000000:1B:00.0 -> 0000:1b:00.0
        node = int(open(f"/sys/bus/pci/devices/{bus.lower()}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def make_decoder(ic, torch, dev, params):
    dec = ic.ColorDecoder(params[0].shape[1], params[0].shape[0], params[4].shape[0]).to(dev)
    with torch.no_grad():
        for p, v in zip(dec.parameters_list(), params):
            p.copy_(torch.tensor(v))
    return dec


def timed_steps(env, step, steps, flush=None):
    """K steps, each bracketed by its own event pair (the optional L2 flush sits between the pairs); returns total ms
    (max over ranks)."""
    torch = env.torch
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    env.barrier()
    for s, e in ev:
        if flush is not None:
            flush.zero_()                   # L2 flush between timed iterations (outside the event pair)
        s.record()
        step()
        e.record()
    env.barrier()
    return env.max_over_ranks(sum(s.elapsed_time(e) for s, e in ev))


def xu_roofline(kernel_ms, clocks, sm_count, npoly, rec):
    """MUFU (XU pipe) roofline of the decode kernel (DESIGN.md section 4): `npoly` of every 8 hidden activations evaluate
    GELU as a polynomial on the FMA pipe, the others cost one MUFU.TANH each; + 2 MUFU (ex2, rcp) per output channel."""
    mhz = (clocks or {}).get("sm_mhz") or (clocks or {}).get("sm_max_mhz")
    ops = 128.0 * (8 - npoly) / 8.0 + 6.0
    out = {"pipe": "xu (MUFU)", "ops_per_texel": ops, "lanes_per_clk_per_sm": 16,
           "ncu_pct_busy_recorded": rec.get("xu_pct_busy"), "recorded_from": rec.get("source")}
    if mhz and kernel_ms:
        peak = sm_count * 16 * mhz * 1e6                      # MUFU results per second
        achieved = ops * SIZE * SIZE / (kernel_ms * 1e-3)
        out.update({"peak_gops": peak / 1e9, "achieved_gops": achieved / 1e9, "frac": achieved / peak, "sm_mhz": mhz})
    return out


def pcie_floor(env, h2d_bytes, d2h_bytes, iters=6):
    """What the box allows: every rank AT ONCE copies h2d_bytes host->device and d2h_bytes device->host per iteration from
    / to pinned memory on two streams (PCIe is full duplex), nothing else running.  Max over ranks."""
    torch = env.torch
    hin = torch.empty(h2d_bytes, dtype=torch.uint8).pin_memory()
    hout = torch.empty(d2h_bytes, dtype=torch.uint8).pin_memory()
    din = torch.empty(h2d_bytes, dtype=torch.uint8, device=env.dev)
    dout = torch.zeros(d2h_bytes, dtype=torch.uint8, device=env.dev)
    s1, s2 = torch.cuda.Stream(device=env.dev), torch.cuda.Stream(device=env.dev)
    res = {}
    for name, do_in, do_out in (("both", True, True), ("h2d_only", True, False), ("d2h_only", False, True)):
        vals = []
        for rep in range(4):                 # the first round warms up; the median of the other three is kept
            env.barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            s1.wait_event(a)
            s2.wait_event(a)
            for _ in range(iters):
                if do_in:
                    with torch.cuda.stream(s1):
                        din.copy_(hin, non_blocking=True)
                if do_out:
                    with torch.cuda.stream(s2):
                        hout.copy_(dout, non_blocking=True)
            main = torch.cuda.current_stream(env.dev)
            main.wait_stream(s1)
            main.wait_stream(s2)
            b.record()
            env.barrier()
            vals.append(env.max_over_ranks(a.elapsed_time(b)) / iters)
        res[name] = sorted(vals[1:])[1]
    return {"ms_per_frame": res["both"], "gtexel_s": env.world * SIZE * SIZE / (res["both"] * 1e-3) / 1e9,
            "h2d_gbs_per_rank": h2d_bytes / (res["h2d_only"] * 1e-3) / 1e9,
            "d2h_gbs_per_rank": d2h_bytes / (res["d2h_only"] * 1e-3) / 1e9,
            "aggregate_gbs": env.world * (h2d_bytes + d2h_bytes) / (res["both"] * 1e-3) / 1e9,
            "what": f"{env.world} rank(s) concurrently: pinned H2D {h2d_bytes} B + D2H {d2h_bytes} B per frame on two streams, no kernels"}


# ------------------------------------------------------------------------------------------------ side benchmarks
def bench_train(args, env, nic, ic, var2):
    """Fused training step at BASELINE config 1 shape: 512^2 image, 8 crops of 256^2 per rank per step (weak DP),
    Philox noise on, the gradient exchange when world > 1, fused Adam + clamp.  `value` INCLUDES the sampling of every
    step (LOD draw on the host, crop origins + target gather on the device: step_sampled); `ms_per_step_presampled` is the
    same step fed from pre-built batches."""
    import inputs as I
    from neural_image_compression_v2_b200 import _lib as L
    torch, dev, world, rank = env.torch, env.dev, env.world, env.rank
    size, nc, crop = 512, 8, 256
    var2.update(IMAGE_SIZE=size)
    fp = [torch.tensor(g, device=dev) for g in I.make_grids(size, 2, seed=3, no_mip=True)]
    dec = make_decoder(ic, torch, dev, I.make_mlp(73, seed=4))
    train_prec = args.train_prec or "f16"
    tr = ic.FusedTrainer(fp, dec, num_epochs=100000, fp_bits=8, seed=1, precision=train_prec, exchange=args.exchange)
    img = I.make_image(size, 2, seed=5)
    img8 = torch.tensor(np.ascontiguousarray(np.floor(np.transpose(img, (1, 2, 0)) * 255 + 0.5).astype(np.uint8)), device=dev)
    pyr = ic.build_mip_pyramid(img8)                   # [3, 512, 512] float32 (TF_NO_MIP: one level)
    imgt = pyr[0]
    g = torch.Generator().manual_seed(100 + rank)
    batches = []
    for _ in range(4):
        coord = torch.randint(0, size - crop + 1, (nc, 2), generator=g)
        batches.append((coord.to(dev), ic.sample_crops(imgt, coord, crop)))
    steps = args.steps
    for i in range(max(args.warmup, 3)):
        tr.step(*batches[i % 4], 0)
        tr.step_sampled(pyr)
    env.barrier()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for i in range(steps):
        tr.step(*batches[i % 4], 0)
    e.record()
    env.barrier()
    ms_pre = env.max_over_ranks(s.elapsed_time(e))
    s.record()
    for i in range(steps):
        loss, _ = tr.step_sampled(pyr)
    e.record()
    env.barrier()
    ms = env.max_over_ranks(s.elapsed_time(e))
    # the training kernel alone, in a second pass: the library's event records around it would sit between the step's
    # kernels and rule out their programmatic (overlapped) launch, so they are kept out of the step timing above
    L.set_option(dev, L.OPT_TIME_KERNELS, 1)
    for i in range(steps):
        tr.step(*batches[i % 4], 0)
    torch.cuda.synchronize()
    kms, kn = L.kernel_time_ms(dev)
    L.set_option(dev, L.OPT_TIME_KERNELS, 0)
    metrics = tr.flush_metrics()
    n = nc * crop * crop
    rate = world * n * steps / (ms * 1e-3) / 1e6
    tf_peak = peaks()[0]
    kernel_tflops = 3 * FLOP_2D * n * kn / (kms * 1e-3) / 1e12 if kms > 0 else None
    exchange = tr.exchange_in_use()
    res = {"value": rate, "unit": "Msamples/s", "samples_per_step": world * n, "ms_per_step": ms / steps,
           "ms_per_step_presampled": ms_pre / steps, "sampling": "inside the timed region (host LOD draw, device-side origins + target gather)",
           "exchange": {"none": "none (1 GPU)", "peer": "fused into Adam over NVLink peer memory (nic_adam_step_exchange)",
                        "sliced": "fused into Adam over NVLink peer memory, sliced (reduce-scatter + all-gather by peer loads / stores)",
                        "nccl": "NCCL all_reduce + Adam", "mixed": "peer + nccl"}[exchange],
           "precision": train_prec, "loss": float(loss), "psnr_8bit_last_step_db": metrics[-1][2] if metrics else None,
           "workload": "train_512x512_8x256x256_crops", "kernel_ms": kms / max(kn, 1), "kernel_tflops": kernel_tflops,
           "roofline_frac": (kernel_tflops / tf_peak) if kernel_tflops else None, "flop_per_sample": 3 * FLOP_2D}
    if world > 1:
        res["replicas_identical"] = replicas_identical(env, [t for t in tr.fp] + [p.detach() for p in dec.parameters_list()])
        res["exchange_timed_out"] = bool(L.exchange_status(dev)) if exchange in ("peer", "sliced", "mixed") else False
    env.barrier()
    tr.close()
    return res


def replicas_identical(env, tensors):
    """True when every rank holds bit-identical copies of `tensors` (max == min of the raw 32-bit patterns over ranks)."""
    torch, dist = env.torch, env.dist
    flat = torch.cat([t.detach().reshape(-1).view(torch.int32) for t in tensors])
    hi, lo = flat.clone(), flat.clone()
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    return bool(torch.equal(hi, lo))


def bench_gather(args, env, nic, ic, var2, fp):
    """K1 alone: materialise X [N, 73] in 16-bit for the whole 4096^2 frame (HBM-write-bound)."""
    import ctypes as C
    from neural_image_compression_v2_b200 import _lib as L
    torch, dev = env.torch, env.dev
    var2.update(IMAGE_SIZE=SIZE)
    n = SIZE * SIZE
    x = torch.empty((n, 73), dtype=torch.float16, device=dev)
    geom = L.make_geom(L.METHOD_2D, fp[0], fp[1], SIZE, 1, -2, 0, 6, L.PE_TRIANGULAR)
    h, lib = L.handle(dev), L.load_library()

    def run():
        L.check(h, lib.nic_gather(h, C.byref(geom), L.ptr(fp[0]), L.ptr(fp[1]), None, L.ptr(x), L.DT_F16, L.stream_ptr(dev)))

    for _ in range(3):
        run()
    torch.cuda.synchronize()
    L.set_option(dev, L.OPT_TIME_KERNELS, 1)
    for _ in range(args.steps):
        run()
    torch.cuda.synchronize()
    kms, kn = L.kernel_time_ms(dev)
    L.set_option(dev, L.OPT_TIME_KERNELS, 0)
    bytes_per_texel = 73 * 2 + 12 * 4 * (1 / 16 + 1 / 64)
    gbs = bytes_per_texel * n * kn / (kms * 1e-3) / 1e9
    hbm = peaks()[1]
    del x
    return {"value": gbs, "unit": "GB/s", "frac_of_hbm_peak": gbs / hbm, "peak": hbm, "kernel_ms": kms / max(kn, 1),
            "bytes_per_texel": bytes_per_texel, "workload": "gather_4096x4096_f16_X", "gtexel_s": n * kn / (kms * 1e-3) / 1e9}


def bench_3d(args, env, nic, ic, var2):
    """General tensor-core decode kernel on the 3-D shapes of BASELINE configs 4 / 5 (side metrics, kernel-only):
    dense 256^3 volume (method 3) and 16.7 M random-access LUT queries (the full-size runs are --workload lut_65 /
    video_1080p120)."""
    import inputs as I
    from neural_image_compression_v2_b200 import _lib as L
    torch, dev = env.torch, env.dev
    size = 256
    var2.update(IMAGE_SIZE=size, IMAGE_DIMENSION=3, COMPRESSION_METHOD=3, CROP_MIP_LEVEL=5)
    fp = [torch.tensor(g, device=dev) for g in I.make_grids(size, 3, seed=2, no_mip=True, quantized=True)]
    dec = make_decoder(ic, torch, dev, I.make_mlp(127, seed=3, gain=2.0))
    out = torch.empty((size, size, size, 3), dtype=torch.uint8, device=dev)
    q = torch.randint(0, size, (1 << 24, 3), device=dev)
    res = {}
    tf_peak = peaks()[0]
    for name, fn, units in (("dense_256^3_method3", lambda: ic.decode(fp, dec, 0, precision=args.prec, out_dtype=torch.uint8, out=out), size ** 3),
                            ("random_access_16.7M_queries", lambda: ic.decode_points(fp, dec, q, 0, precision=args.prec, out_dtype=torch.uint8), q.shape[0])):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        L.set_option(dev, L.OPT_TIME_KERNELS, 1)
        for _ in range(args.steps):
            fn()
        torch.cuda.synchronize()
        kms, kn = L.kernel_time_ms(dev)
        L.set_option(dev, L.OPT_TIME_KERNELS, 0)
        rate = units * kn / (kms * 1e-3)
        res[name] = {"value": rate / 1e9, "unit": "Gtexel/s", "kernel_ms": kms / max(kn, 1),
                     "roofline_frac": rate * FLOP_M3 / 1e12 / tf_peak}
    var2.update(IMAGE_SIZE=SIZE, IMAGE_DIMENSION=2, COMPRESSION_METHOD=1)
    return res


# ------------------------------------------------------------------------------------------------ headline workload
def run_decode_4096(args, env):
    import neural_image_compression_v2_b200 as nic
    from neural_image_compression_v2_b200 import _lib as L
    from neural_image_compression_v2_b200 import image_compression as ic
    from neural_image_compression_v2_b200 import fp_def, var2
    torch, dev, world, rank = env.torch, env.dev, env.world, env.rank
    var2.update(IMAGE_SIZE=SIZE)
    grids, params = synthetic_model(seed=rank)             # one frame per rank (frame-sharded decode, no collective)
    fp = [torch.tensor(g, device=dev) for g in grids]
    dec = make_decoder(ic, torch, dev, params)
    out = torch.empty((SIZE, SIZE, 3), dtype=torch.uint8, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # > 126 MB L2
    texels = SIZE * SIZE
    tf_peak, hbm_peak, src = peaks()

    def measure(prec, keep_frame=False):
        session = ic.DecodeSession(fp, dec, precision=prec)      # tables (re-packed weights) built once per model
        for _ in range(args.warmup):
            flush.zero_()
            session.decode(0, out_dtype=torch.uint8, out=out)
        env.barrier()
        l0 = nic.launch_count(dev)
        L.set_option(dev, L.OPT_TIME_KERNELS, 1)
        ms = timed_steps(env, lambda: session.decode(0, out_dtype=torch.uint8, out=out), args.steps, flush)
        frame = out.cpu().numpy() if keep_frame else None        # the last timed step's frame, before other legs reuse `out`
        kms, kn = L.kernel_time_ms(dev)
        L.set_option(dev, L.OPT_TIME_KERNELS, 0)
        launches = nic.launch_count(dev) - l0
        # the same step when the model's tables are rebuilt on every call (plain `decode`)
        ms_b = timed_steps(env, lambda: ic.decode(fp, dec, 0, precision=prec, out_dtype=torch.uint8, out=out), args.steps, flush)
        return {"ms_per_step": ms / args.steps, "kernel_ms": kms / max(kn, 1), "launches": launches,
                "value": world * texels / (ms / args.steps * 1e-3) / 1e9,
                "value_with_table_build": world * texels / (ms_b / args.steps * 1e-3) / 1e9, "frame": frame}

    sampler = ClockSampler(env.local) if rank == 0 else None
    main = measure(args.prec, keep_frame=bool(args.dump_outputs) and rank == 0)
    clocks = sampler.stop() if sampler else None
    other = "bf16" if args.prec == "f16" else "f16"
    alt = measure(other) if args.prec != "f32" else None
    # leave the resident frame of the headline precision in `out` (compared with the e2e frame and the CPU reference)
    ic.decode(fp, dec, 0, precision=args.prec, out_dtype=torch.uint8, out=out)

    # ---- e2e: host buffers in, host buffer out, through the public API
    codes = [c.cpu().pin_memory() for c in fp_def.fp_savable(fp, 8)]
    host_params = [p.detach().cpu().pin_memory() for p in dec.parameters_list()]
    host_out = torch.empty((SIZE, SIZE, 3), dtype=torch.uint8).pin_memory()
    h2d = sum(c.numel() for c in codes) + sum(p.numel() * 4 for p in host_params)
    d2h = host_out.numel()
    pipe = ic.HostDecodePipeline(SIZE, dev, precision=args.prec, bands=args.e2e_bands)

    def e2e_step():
        pipe.decode_frame(codes, host_params, host_out, wait=False)      # D2H of frame i overlaps frame i + 1

    for _ in range(3):
        e2e_step()
    pipe.finish()
    env.barrier()
    k2 = args.steps                          # the same K steps as `value`; pipeline fill and drain are inside the timed region
    # Three timed regions of K steps each, the MEDIAN reported and all three listed: the copies share the host's PCIe root
    # and memory with whatever else runs on the box, and a 20 ms region is short enough to be hit by one transient.
    e2e_runs = []
    for _ in range(3):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(k2):
            e2e_step()
        pipe.finish()                        # every frame of the timed region is in host memory before the stop event
        e.record()
        env.barrier()
        e2e_runs.append(env.max_over_ranks(s.elapsed_time(e)) / k2)
    e2e_ms = sorted(e2e_runs)[1]
    e2e_value = world * texels / (e2e_ms * 1e-3) / 1e9
    e2e_ok = bool(torch.equal(host_out.to(dev), out))
    floor = pcie_floor(env, h2d, d2h)
    out_host = out.cpu().numpy() if rank == 0 else None

    extras = {}
    if not args.no_extras:
        extras["gather"] = bench_gather(args, env, nic, ic, var2, fp)
        del fp, out, flush
        extras["decode_3d"] = bench_3d(args, env, nic, ic, var2)
        extras["train"] = bench_train(args, env, nic, ic, var2)

    if rank == 0:
        kms = main["kernel_ms"]
        sm_count = torch.cuda.get_device_properties(dev).multi_processor_count
        achieved = FLOP_2D * texels / (kms * 1e-3) / 1e12
        rec = recorded_profile("decode_tc2d_ws_kernel")
        npoly = 3
        cfg = decode_config()
        line = {
            "metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.prec, "data": "synthetic", "config": cfg,
            "notes": {"frames_per_step": world, "l2": "flushed between timed iterations (256 MB write)",
                      "tables": "`value`: the model's private tensor-core tables (16-bit shadow grids, G1 rows, packed weights) are "
                                "built once per MODEL (DecodeSession) and amortised over its frames, like any weight pre-packing; "
                                "`value_with_table_build` rebuilds them every step (one-shot texture); e2e receives a new model "
                                "from the host every step and always rebuilds"},
            "value_with_table_build": main["value_with_table_build"],
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": tf_peak, "unit": "TFLOP/s", "frac": achieved / tf_peak,
                         "traffic": rec.get("traffic_bytes"), "traffic_recorded_from": rec.get("source"),
                         "peak_source": f"{src} bf16_tflops (burst: kernel timed alone)",
                         "flop_per_texel": FLOP_2D, "kernel": "decode_tc2d_ws_kernel", "kernel_ms": kms,
                         "kernel_share_of_step": kms / main["ms_per_step"],
                         "tensor_pct_active_recorded": rec.get("tensor_pct_active"),
                         # tools/ubench/mma_rate2.cu: an SS-form M128 x N64 x K16 tcgen05.mma (hidden width 64) holds the
                         # tensor pipe 48.1 cycles (shared-memory operand fetch) for 32 cycles of math
                         "attainable_frac_ss_form_hidden_64": 32.0 / 48.1,
                         "binding_pipe": xu_roofline(kms, clocks, sm_count, npoly, rec)},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_frame": e2e_ms, "ms_per_frame_runs": e2e_runs, "timing": "median of three timed regions of K steps",
                    "matches_resident_output": e2e_ok, "pcie_floor": floor,
                    "frac_of_pcie_floor": floor["ms_per_frame"] / e2e_ms},
            "gpu_launches": int(main["launches"]), "clocks": clocks, "numa_node_rank0": env.numa,
        }
        if alt:
            a_ach = FLOP_2D * texels / (alt["kernel_ms"] * 1e-3) / 1e12
            line[other] = {"value": alt["value"], "unit": UNIT, "ms_per_step": alt["ms_per_step"], "kernel_ms": alt["kernel_ms"],
                           "value_with_table_build": alt["value_with_table_build"], "roofline_frac": a_ach / tf_peak}
        line.update(extras)
        if world == 1 and not args.no_cpu:
            threads = os.cpu_count() or 1
            ctx = cpu_setup(threads)
            keep = {}
            cpu_decode_tiles(ctx, 1)
            done, dt = cpu_decode_tiles(ctx, args.cpu_baseline_tiles, 0, keep)
            line["cpu_baseline"] = {"value": done / dt / 1e9, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": f"{args.cpu_baseline_tiles} tiles of {CPU_TILE}x{CPU_TILE} texels ({dt:.1f} s), torch-CPU "
                                              "port of the reference op sequence (oracle/nic_oracle_torch.py)"}
            line["psnr"] = psnr_vs_reference(out_host, keep)
            if "train" in line:
                line["train"]["cpu_value"] = cpu_train_rate(threads)
        if args.dump_outputs:
            dump_frame_sample(args.dump_outputs, main["frame"])
        env.emit(line)


DUMP_TEXELS = 1 << 22            # 4.2 M of the 16.8 M texels: 48 MB as float32


def dump_frame_sample(out_dir, frame):
    """Writes DIR/frame.npy: the uint8 RGB values of a fixed, seeded sample of the last timed step's 4096^2 frame, as
    float32 [DUMP_TEXELS, 3], texels in raster order (row-major flat index).  The inputs are seeded too, so two builds run
    with the same arguments can be compared value for value."""
    idx = np.sort(np.random.default_rng(0).choice(SIZE * SIZE, DUMP_TEXELS, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "frame.npy"), frame.reshape(-1, 3)[idx].astype(np.float32))


def psnr_vs_reference(ours_u8, ref_tiles):
    """The metric's "PSNR vs reference": the tensor-core frame against the fp32 reference frame (CPU port of the reference op
    sequence), 8-bit images, reference formula 10 log10(256^2 / mse) (utils.py:117-130), over the tiles the CPU leg decoded."""
    n = SIZE // CPU_TILE
    sse, cnt, within1, exact = 0.0, 0, 0, 0
    for i, ref in ref_tiles.items():
        x, y = i % n, i // n
        t = ours_u8[CPU_TILE * x:CPU_TILE * (x + 1), CPU_TILE * y:CPU_TILE * (y + 1)].astype(np.int32)
        d = np.abs(t - ref.astype(np.int32))
        sse += float(np.sum(d.astype(np.float64) ** 2))
        cnt += d.size
        within1 += int((d <= 1).sum())
        exact += int((d == 0).sum())
    mse = sse / max(cnt, 1)
    return {"vs_reference_db": float("inf") if mse == 0 else 10 * np.log10(65536.0 / mse), "within_1_lsb": within1 / max(cnt, 1),
            "exact": exact / max(cnt, 1), "texels": cnt // 3, "formula": "10 log10(256^2 / mse) on 8-bit frames (utils.py:117-130)",
            "tolerance": ">= 99.9 % within +-1 LSB (north star)"}


# ------------------------------------------------------------------------------------------------ config 2, strong scaling
def run_decode_strong(args, env):
    """ONE 4096^2 frame tiled across the N GPUs (BASELINE config 2 "tiled across 1/2/4/8 B200"): rank r decodes the row
    band parallel.shard_rows gives it (parallel.decode_band), no collective; time = max over ranks."""
    from neural_image_compression_v2_b200 import _lib as L
    from neural_image_compression_v2_b200 import image_compression as ic
    from neural_image_compression_v2_b200 import parallel, var2
    torch, dev, world, rank = env.torch, env.dev, env.world, env.rank
    var2.update(IMAGE_SIZE=SIZE)
    grids, params = synthetic_model(seed=0)                # the SAME model on every rank
    fp = [torch.tensor(g, device=dev) for g in grids]
    dec = make_decoder(ic, torch, dev, params)
    r0, rows = parallel.shard_rows(SIZE, rank, world)
    band = torch.empty((rows, SIZE, 3), dtype=torch.uint8, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    session = ic.DecodeSession(fp, dec, precision=args.prec)

    def step():
        session.decode(0, size=(rows, SIZE), origin=(r0, 0), out_dtype=torch.uint8, out=band)

    for _ in range(args.warmup):
        flush.zero_()
        step()
    L.set_option(dev, L.OPT_TIME_KERNELS, 1)
    ms = timed_steps(env, step, args.steps, flush) / args.steps
    kms, kn = L.kernel_time_ms(dev)
    L.set_option(dev, L.OPT_TIME_KERNELS, 0)
    full = ic.decode(fp, dec, 0, precision=args.prec, out_dtype=torch.uint8)
    ok = torch.tensor([int(torch.equal(full[r0:r0 + rows], band))], device=dev)
    if world > 1:
        env.dist.all_reduce(ok, op=env.dist.ReduceOp.MIN)
    tf_peak = peaks()[0]
    value = SIZE * SIZE / (ms * 1e-3) / 1e9
    env.emit({"metric": "decoded Gtexel/s (ONE 4096x4096 RGB frame tiled over the GPUs)", "value": value, "unit": UNIT,
              "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
              "scaling": "strong", "vs_baseline": None, "dtype": args.prec, "data": "synthetic",
              "config": {"workload": "decode_4096x4096_rgb_strong", "rows_per_rank": rows, "l2": "flushed between timed iterations"},
              "bands_equal_full_frame": bool(ok.item()),
              "roofline": {"bound": "tensor", "achieved": value * FLOP_2D / 1e3, "peak": tf_peak * world, "unit": "TFLOP/s",
                           "frac": value * FLOP_2D / 1e3 / (tf_peak * world), "kernel_ms_rank0": kms / max(kn, 1), "traffic": None}})


# ------------------------------------------------------------------------------------------------ config 3
def run_train_2048(args, env):
    """BASELINE config 3: a 2048^2 multi-channel material texture stack (9 channels) with mip levels 0..11, data-parallel
    training on the tensor-core path, 8 crops per rank per step, LOD drawn per step with the reference's distribution
    (the same on every rank), device-side sampling inside the timed region.  Level 0's flat gradient buffer is 15.8 MB:
    above FusedTrainer.PEER_EXCHANGE_MAX_BYTES, so with more than two ranks its exchange runs sliced inside the Adam kernel
    (`--exchange nccl` times the NCCL all-reduce baseline instead); smaller levels use the one-shot fused exchange."""
    from neural_image_compression_v2_b200 import _lib as L
    from neural_image_compression_v2_b200 import image_compression as ic
    from neural_image_compression_v2_b200 import fp_def, var2
    torch, dev, world, rank = env.torch, env.dev, env.world, env.rank
    size, cout, nc = 2048, 9, 8
    var2.update(IMAGE_SIZE=size, TF_NO_MIP=False, MAX_MIP_LEVEL=11, NUM_CROPS=nc, OUTPUT_CHANNELS=cout)
    g = torch.Generator(device=dev).manual_seed(7)
    yy, xx = torch.meshgrid(torch.arange(size, device=dev) / size, torch.arange(size, device=dev) / size, indexing="ij")
    chans = []
    for c in range(cout):
        f = torch.rand(4, generator=g, device=dev) * 5 + 0.5
        v = 127.5 + 50 * (torch.sin(6.2832 * (f[0] * xx + f[1] * yy)) + torch.sin(6.2832 * (f[2] * xx - f[3] * yy)))
        chans.append(v + (torch.rand(size, size, generator=g, device=dev) - 0.5) * 16)
    img8 = torch.stack(chans, dim=-1).clamp(0, 255).round().to(torch.uint8).contiguous()
    pyr = ic.build_mip_pyramid(img8)                                   # 12 mips, [9, S, S] float32 each
    torch.manual_seed(11)                                              # identical initial replicas
    fp, levels = fp_def.create_pyramid(size // 4, 12, 8, dev, torch.float32)
    fp = [p.detach() for p in fp]
    dec = ic.ColorDecoder(73, 64, cout).to(dev)
    prec = args.train_prec or "bf16"                                   # config 3 names bf16
    tr = ic.FusedTrainer(fp, dec, num_epochs=1000000, fp_bits=8, seed=3, precision=prec, exchange=args.exchange)
    steps = args.steps
    for _ in range(max(args.warmup, 20)):                              # touches most levels (peer buffers are mapped on first use)
        tr.step_sampled(pyr)
    env.barrier()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    samples, lods = 0, []
    s.record()
    t_host = time.perf_counter()
    for _ in range(steps):
        _, lod = tr.step_sampled(pyr)
        lods.append(lod)
        samples += nc * (max(1, 256 >> lod)) ** 2
    t_host = time.perf_counter() - t_host
    e.record()
    env.barrier()
    ms = env.max_over_ranks(s.elapsed_time(e))
    host_ms = env.max_over_ranks(1e3 * t_host) / steps                 # enqueue time of a step (no sync inside the loop)
    metrics = tr.flush_metrics()
    ident = replicas_identical(env, list(tr.fp) + [p.detach() for p in dec.parameters_list()]) if world > 1 else None
    tf_peak = peaks()[0]
    flop = 3 * 2 * (73 * 64 + 64 * 64 + 64 * cout)
    value = world * samples / (ms * 1e-3) / 1e6
    exchange = tr.exchange_in_use()
    timed_out = bool(L.exchange_status(dev)) if exchange in ("peer", "sliced", "mixed") else False
    env.emit({"metric": "train Msamples/s (2048^2 x 9-channel material stack with mips, data parallel)", "value": value,
              "unit": "Msamples/s", "n_gpus": world, "steps": steps, "warmup": max(args.warmup, 20), "ms_per_step": ms / steps,
              "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": prec, "data": "synthetic",
              "config": {"workload": "train_2048x2048x9_mips0-11", "crops_per_rank": nc, "crop": "256 >> lod", "levels": levels,
                         "flat_gradient_bytes_level0": 4 * (fp[0].numel() + fp[1].numel() + sum(p.numel() for p in dec.parameters_list())),
                         "sampling": "inside the timed region"},
              "samples_timed_per_rank": samples, "lod_histogram": {str(k): lods.count(k) for k in sorted(set(lods))},
              "exchange": exchange, "exchange_timed_out": timed_out, "replicas_identical": ident,
              "host_enqueue_ms_per_step": host_ms,
              "loss_last": metrics[-1][1] if metrics else None, "psnr_8bit_last_step_db": metrics[-1][2] if metrics else None,
              "roofline": {"bound": "tensor", "achieved": value * flop / 1e6, "peak": tf_peak * world, "unit": "TFLOP/s",
                           "frac": value * flop / 1e6 / (tf_peak * world), "flop_per_sample": flop, "traffic": None,
                           "note": "whole step (sampler, prep, training kernel, finish, exchange, Adam), not the kernel alone"}})
    env.barrier()
    tr.close()


# ------------------------------------------------------------------------------------------------ config 4
def run_lut_65(args, env):
    """BASELINE config 4: a 65^3 RGB colour LUT (grids with one extra node per axis: 18^3 / 10^3, SURVEY 8(d)), random-access
    decode of 1e9 query points in chunks of 2^25, queries sharded over the ranks (no collective)."""
    from neural_image_compression_v2_b200 import _lib as L
    from neural_image_compression_v2_b200 import image_compression as ic
    from neural_image_compression_v2_b200 import parallel, var2
    import inputs as I
    torch, dev, world, rank = env.torch, env.dev, env.world, env.rank
    var2.update(IMAGE_SIZE=64, IMAGE_DIMENSION=3, COMPRESSION_METHOD=3, CROP_MIP_LEVEL=3)
    rng = np.random.default_rng(94)
    lo, hi = I.q_range(8)
    grids = [rng.uniform(lo, hi, (12, 18, 18, 18)).astype(np.float32), rng.uniform(lo, hi, (12, 10, 10, 10)).astype(np.float32)]
    grids = [(np.floor(g * np.float32(255) + np.float32(0.5)) / np.float32(255)).astype(np.float32) for g in grids]
    fp = [torch.tensor(g, device=dev) for g in grids]
    from neural_image_compression_v2_b200 import fp_def
    codes = fp_def.fp_savable(fp, 8)                       # the deployment form of the LUT: uint8 codes (82 KB)
    dec = make_decoder(ic, torch, dev, I.make_mlp(127, seed=95, gain=2.0))
    table = {0: 0}
    total = int(args.queries)
    q0, q1 = parallel.shard_range(total, rank, world)
    chunk = 1 << 25
    gen = torch.Generator(device=dev).manual_seed(1 + rank)
    qs = [torch.randint(0, 65, (chunk, 3), generator=gen, device=dev) for _ in range(4)]      # 4 distinct chunks, cycled
    mine = q1 - q0
    sizes = [chunk] * (mine // chunk) + ([mine % chunk] if mine % chunk else [])

    def step():
        for i, n in enumerate(sizes):
            ic.decode_points_codes(codes, dec, qs[i % 4][:n], 8, 0, precision=args.prec, out_dtype=torch.uint8, level_table=table)

    for _ in range(min(args.warmup, 2)):
        step()
    steps = args.steps
    L.set_option(dev, L.OPT_TIME_KERNELS, 1)
    ms = timed_steps(env, step, steps) / steps
    kms, kn = L.kernel_time_ms(dev)
    L.set_option(dev, L.OPT_TIME_KERNELS, 0)
    # parity of the timed path: the first chunk's answers equal the dense decode of the LUT at those coordinates
    dense = ic.decode(fp, dec, 0, size=65, precision=args.prec, out_dtype=torch.uint8, level_table=table)
    pts = ic.decode_points_codes(codes, dec, qs[0][:1 << 20], 8, 0, precision=args.prec, out_dtype=torch.uint8, level_table=table)
    c = qs[0][:1 << 20]
    want = dense[c[:, 0], c[:, 1], c[:, 2]].to(torch.int32)
    dd = (pts.to(torch.int32) - want).abs()
    ok = {"within_1_lsb": float((dd <= 1).float().mean()), "exact": float((dd == 0).float().mean()), "max": int(dd.max())}
    # ... and the same queries on the general kernel (grids in global memory), for reference
    L.set_option(dev, L.OPT_DISABLE_FAST2D, 1)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ic.decode_points_codes(codes, dec, qs[0], 8, 0, precision=args.prec, out_dtype=torch.uint8, level_table=table)
    t0.record()
    for i in range(4):
        ic.decode_points_codes(codes, dec, qs[i], 8, 0, precision=args.prec, out_dtype=torch.uint8, level_table=table)
    t1.record()
    torch.cuda.synchronize()
    general_rate = 4 * chunk / (t0.elapsed_time(t1) * 1e-3) / 1e9
    L.set_option(dev, L.OPT_DISABLE_FAST2D, 0)
    tf_peak = peaks()[0]
    value = total / (ms * 1e-3) / 1e9
    env.emit({"metric": "random-access decoded Gquery/s (65^3 RGB LUT, 1e9 queries)", "value": value, "unit": "Gquery/s",
              "n_gpus": world, "steps": steps, "warmup": min(args.warmup, 2), "ms_per_step": ms, "higher_is_better": True,
              "scaling": "strong", "vs_baseline": None, "dtype": args.prec, "data": "synthetic",
              "config": {"workload": "lut_65^3_random_access", "queries_per_step": total, "chunk": chunk,
                         "model": "uint8 codes of an 18^3 + 10^3-node grid pair (82 KB) + 127-64-64-3 decoder",
                         "inputs": "int64 [Q, 3] coordinates resident in HBM (4 distinct chunks per rank, cycled)"},
              "points_vs_dense_decode": ok, "general_kernel_gquery_s_per_gpu": general_rate,
              "roofline": {"bound": "tensor", "achieved": value * FLOP_M3 / 1e3, "peak": tf_peak * world, "unit": "TFLOP/s",
                           "frac": value * FLOP_M3 / 1e3 / (tf_peak * world), "kernel_ms_per_step_rank0": kms / steps if kn else None,
                           "kernel": "decode_codes_smem_kernel<3> (grids resident in shared memory as uint8 codes)" if args.prec == "f16"
                           else "decode_tc_gws_kernel<3> (queries)", "traffic": None}})


# ------------------------------------------------------------------------------------------------ config 5
def run_video(args, env):
    """BASELINE config 5: a 1920x1080x120-frame video volume on (x, y, t) grids (method 3), frame-sharded decode: rank r
    decodes frames [f0, f1) of the 120 (parallel.decode_slab), grids replicated, no collective."""
    from neural_image_compression_v2_b200 import _lib as L
    from neural_image_compression_v2_b200 import image_compression as ic
    from neural_image_compression_v2_b200 import parallel, var2
    import inputs as I
    torch, dev, world, rank = env.torch, env.dev, env.world, env.rank
    var2.update(IMAGE_SIZE=2048, IMAGE_DIMENSION=3, COMPRESSION_METHOD=3, CROP_MIP_LEVEL=5)
    vol = (120, 1080, 1920)                                # (t, y, x): the first axis is the frame axis
    lo, hi = I.q_range(8)
    gen = torch.Generator(device=dev).manual_seed(5)

    def grid(div):
        shape = (12, vol[2] // div + 1, vol[1] // div + 1, vol[0] // div + 1)      # [C, z, y, x], x = first image axis
        g = torch.rand(shape, generator=gen, device=dev) * (hi - lo) + lo
        return (torch.floor(g * 255 + 0.5) / 255).contiguous()

    fp = [grid(4), grid(8)]
    dec = make_decoder(ic, torch, dev, I.make_mlp(127, seed=6, gain=2.0))
    table = {0: 0}
    f0, f1 = parallel.shard_range(vol[0], rank, world)
    out = torch.empty((f1 - f0, vol[1], vol[2], 3), dtype=torch.uint8, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def step():
        if f1 > f0:
            ic.decode(fp, dec, 0, size=(f1 - f0, vol[1], vol[2]), origin=(f0, 0, 0), precision=args.prec, out_dtype=torch.uint8,
                      out=out, level_table=table)

    for _ in range(args.warmup):
        step()
    steps = args.steps
    L.set_option(dev, L.OPT_TIME_KERNELS, 1)
    ms = timed_steps(env, step, steps, flush) / steps
    kms, kn = L.kernel_time_ms(dev)
    L.set_option(dev, L.OPT_TIME_KERNELS, 0)
    # parity of the timed path: one 64^3 sub-cube of this rank's slab against the fp32 reference-exact kernel
    ok = None
    if f1 - f0 >= 8:
        n0 = min(64, f1 - f0)
        ref = ic.decode(fp, dec, 0, size=(n0, 64, 64), origin=(f0, 512, 960), precision="f32", out_dtype=torch.uint8, level_table=table)
        d = (out[:n0, 512:576, 960:1024].to(torch.int32) - ref.to(torch.int32)).abs()
        ok = float((d <= 1).float().mean())
    texels = vol[0] * vol[1] * vol[2]
    tf_peak = peaks()[0]
    value = texels / (ms * 1e-3) / 1e9
    env.emit({"metric": "decoded Gtexel/s (1920x1080x120 video volume, frame-sharded)", "value": value, "unit": UNIT,
              "n_gpus": world, "steps": steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
              "scaling": "strong", "vs_baseline": None, "dtype": args.prec, "data": "synthetic",
              "config": {"workload": "video_1920x1080x120_method3", "frames_per_rank": f1 - f0, "grids": [list(g.shape) for g in fp],
                         "output": "uint8", "l2": "flushed between timed iterations"},
              "within_1_lsb_of_f32_kernel_on_64^3_subcube": ok,
              "roofline": {"bound": "tensor", "achieved": value * FLOP_M3 / 1e3, "peak": tf_peak * world, "unit": "TFLOP/s",
                           "frac": value * FLOP_M3 / 1e3 / (tf_peak * world), "kernel_ms_rank0": kms / max(kn, 1) if kn else None,
                           "kernel": "decode_tc_gws_kernel<3>", "traffic": None}})


WORKLOADS = {"decode_4096": run_decode_4096, "decode_4096_strong": run_decode_strong, "train_2048_mips": run_train_2048,
             "lut_65": run_lut_65, "video_1080p120": run_video}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="decode_4096", choices=sorted(WORKLOADS))
    ap.add_argument("--prec", default="f16", choices=["f16", "bf16", "f32"])
    ap.add_argument("--train-prec", default=None, choices=["f16", "bf16", "f32"],
                    help="training precision (default: f16 for the config-1 side benchmark, bf16 for train_2048_mips)")
    ap.add_argument("--queries", type=float, default=1e9, help="lut_65: query points per step")
    ap.add_argument("--cpu-baseline-tiles", type=int, default=48,
                    help="cpu_baseline leg: 1024^2 tiles decoded on the host cores (48 = three frames, ~10 s on 16 cores)")
    ap.add_argument("--e2e-bands", type=int, default=4, help="row bands per frame of the host-to-host pipeline")
    ap.add_argument("--exchange", default="auto", choices=["auto", "nccl", "peer", "sliced"],
                    help="training workloads at N > 1: the data-parallel exchange (FusedTrainer)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the gather, 3-D and training side benchmarks")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="decode_4096: after the timed steps, write a seeded sample of the last step's frame to DIR/frame.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "decode_4096"):
        ap.error("--dump-outputs covers the decode_4096 workload of --impl ours")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
        return
    env = Env()
    try:
        WORKLOADS[args.workload](args, env)
    finally:
        env.close()


if __name__ == "__main__":
    main()
