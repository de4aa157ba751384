"""Filtered sampling at continuous coordinates (nic_sample / nic_sample_codes, image_compression.sample*): the tap rule's
oracle against torch's grid_sample, the ABI of NicSampler, and on the GPU the fp32 arm against the oracle, the tensor-core
arm against the fp32 arm and against its own unfused composition, decode-from-codes, mip blending and table reuse."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

import inputs as I
from helpers import T, configure, dev, lsb_stats, make_decoder, psnr256
from sample_oracle import blend_lod, sample_filtered, tap_rule

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def nic():
    import neural_image_compression_v2_b200 as n
    return n


def dyadic_coords(rng, q, dim):
    """Coordinates k / 256 in [-1, 2): inside, on and outside [0, 1]; every product with an integer extent is exact, so the
    oracle's taps and weights equal grid_sample's."""
    c = rng.integers(-256, 512, (q, dim)).astype(np.float32) / np.float32(256)
    c[:4] = [[0.0] * dim, [1.0] * dim, [-0.5] * dim, [1.5] * dim]
    return c


# ------------------------------------------------------------------------------------------------ no GPU
@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("align_corners", [False, True])
def test_oracle_equals_grid_sample_border(dim, align_corners):
    rng = np.random.default_rng(300 + dim)
    extent = (13, 8) if dim == 2 else (7, 5, 9)
    dense = rng.random(extent + (3,))                                    # [Sx, Sy(, Sz), C], x the first (slow) axis
    coords = dyadic_coords(rng, 997, dim)
    got = sample_filtered(dense, coords, align_corners, "clamp")
    # grid_sample: input [N, C, (D,) H, W] with W indexed by grid[..., 0]; our x axis is W, y is H, z is D
    inp = torch.tensor(dense).permute(*range(dim, -1, -1)).unsqueeze(0)
    g = torch.tensor(coords, dtype=torch.float64) * 2 - 1
    grid = g.reshape((1, -1) + (1,) * (dim - 1) + (dim,))
    want = torch.nn.functional.grid_sample(inp, grid, mode="bilinear", padding_mode="border", align_corners=align_corners)
    want = want.reshape(3, -1).T.numpy()
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-6)


@pytest.mark.parametrize("align_corners", [False, True])
def test_oracle_wrap_equals_a_modular_loop(align_corners):
    rng = np.random.default_rng(310)
    dense = rng.random((6, 5, 4, 2))
    coords = dyadic_coords(rng, 301, 3)
    got = sample_filtered(dense, coords, align_corners, "wrap")
    for q in range(coords.shape[0]):
        acc = np.zeros(2)
        axes = []
        for a in range(3):
            s = dense.shape[a]
            p = coords[q, a] * (s - 1) if align_corners else coords[q, a] * s - 0.5
            i0 = int(np.floor(p))
            axes.append([(i0 % s, 1 - (p - i0)), ((i0 + 1) % s, p - i0)])
        for (ix, wx) in axes[0]:
            for (iy, wy) in axes[1]:
                for (iz, wz) in axes[2]:
                    acc += wx * wy * wz * dense[ix, iy, iz]
        np.testing.assert_allclose(got[q], acc, rtol=0, atol=1e-6)


def test_tap_rule_edge_cases():
    """NaN maps to -2^24 (the first texel under clamp), huge coordinates stay finite, weights sum to one."""
    c = np.array([[np.nan, 0.5], [1e30, -1e30], [0.25, 0.75]], np.float32)
    taps, w = tap_rule(c, (16, 8), False, "clamp")
    assert (taps[0, :, 0] == 0).all() and (taps[1, :, 0] == 15).all() and (taps[1, :, 1] == 0).all()
    np.testing.assert_allclose(w.sum(1), 1.0, atol=1e-6)
    taps, w = tap_rule(c, (16, 8), False, "wrap")
    assert ((taps >= 0) & (taps < np.array([16, 8]))).all()


def test_sampler_struct_layout_matches_the_binding(tmp_path):
    L = nic()._lib
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "nic.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(NicSampler));']
    for field, _ in L.NicSampler._fields_:
        lines.append(f'  printf("{field} %zu\\n", offsetof(NicSampler, {field}));')
    lines += ['  printf("clamp %d wrap %d\\n", NIC_ADDRESS_CLAMP, NIC_ADDRESS_WRAP);', '  return 0;', '}']
    src = tmp_path / "sampler.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "sampler"
    subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split("\n")
    got = {l.split()[0]: int(l.split()[1]) for l in out if l.strip() and not l.startswith("clamp")}
    assert got["size"] == ctypes.sizeof(L.NicSampler)
    for field, _ in L.NicSampler._fields_:
        assert got[field] == getattr(L.NicSampler, field).offset, field
    assert [l for l in out if l.startswith("clamp")] == [f"clamp {L.ADDRESS_CLAMP} wrap {L.ADDRESS_WRAP}"]


def test_host_checks_of_the_coordinates():
    """dtype and layout of coords are checked before anything is launched; host tensors are refused (no CPU fallback)."""
    n = nic()
    ic = n.image_compression
    configure()
    dec = ic.ColorDecoder(in_channels=73, hidden=64, out_channels=3)
    fp = [torch.zeros(12, 129, 129), torch.zeros(12, 65, 65)]
    with pytest.raises(TypeError):
        ic.sample(fp, dec, torch.zeros((4, 2), dtype=torch.int64))
    with pytest.raises(TypeError):
        ic.sample(fp, dec, torch.zeros((2, 4), dtype=torch.float32).T)
    with pytest.raises(ValueError):
        ic.sample(fp, dec, torch.zeros((4, 3), dtype=torch.float32))
    with pytest.raises(n.NicError):
        ic.sample(fp, dec, torch.zeros((4, 2), dtype=torch.float32))
    with pytest.raises(ValueError):
        ic.sample(fp, dec, torch.zeros((4, 2), dtype=torch.float32), lod=0.5, size=64)


# ------------------------------------------------------------------------------------------------ GPU
def query_coords(rng, q, dim):
    """Random coordinates in [-0.25, 1.25) with 0, 1, points outside [0, 1] and NaN among them."""
    c = (rng.random((q, dim), dtype=np.float32) * np.float32(1.5) - np.float32(0.25)).astype(np.float32)
    c[:6] = [[0.0] * dim, [1.0] * dim, [-0.3] * dim, [1.7] * dim, [np.nan] * dim, [0.5] * dim]
    c[6, 0] = np.nan
    return c


_MODELS = {}


def model(kind):
    """(grids, params, table, method, mip, extent) of a test model and the oracle's dense frame of that mip (cached)."""
    if kind in _MODELS:
        return _MODELS[kind]
    from oracle import nic_oracle as O
    if kind.startswith("2d"):
        size, mip = 64, (0 if kind == "2d_mip0" else 3)       # mip 3 on pyramid level 0: step 2, G1 interpolation off
        grids = I.make_grids(size, 2, seed=320, quantized=True)
        params = I.make_mlp(73, seed=321, gain=2.0)
        table = O.create_pyramid_mip_levels(size, size // 4)
        method, extent = 1, size >> mip
    else:
        method = 3 if kind == "3d_m3" else 4
        rng = np.random.default_rng(322 + method)
        lo, hi = I.q_range(8)
        grids = [rng.uniform(lo, hi, (12, 10, 10, 10)).astype(np.float32), rng.uniform(lo, hi, (12, 6, 6, 6)).astype(np.float32)]
        params = I.make_mlp(127 if method == 3 else 79, seed=323, gain=2.0)
        table, mip, extent = {0: 0}, 0, 33
    dense = O.decode_block(grids, params, extent, mip, table, method, use_tri_pe=True)
    _MODELS[kind] = (grids, params, table, method, mip, extent, dense)
    return _MODELS[kind]


def setup(kind):
    grids, params, table, method, mip, extent, dense = model(kind)
    if method == 1:
        configure(IMAGE_SIZE=64, TF_NO_MIP=False, MAX_MIP_LEVEL=6)
    else:
        configure(IMAGE_SIZE=64, IMAGE_DIMENSION=3, COMPRESSION_METHOD=method)
    return [T(g) for g in grids], make_decoder(params), table, method, mip, extent, dense


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["2d_mip0", "2d_mip3", "3d_m3", "3d_m4"])
@pytest.mark.parametrize("address", ["clamp", "wrap"])
@pytest.mark.parametrize("align_corners", [False, True])
def test_f32_sample_equals_oracle(kind, address, align_corners):
    ic = nic().image_compression
    fp, dec, table, method, mip, extent, dense = setup(kind)
    dim = 2 if method == 1 else 3
    rng = np.random.default_rng(330)
    c = query_coords(rng, 1003, dim)                                      # not a multiple of 32
    got = ic.sample(fp, dec, T(c), mip, extent, address=address, align_corners=align_corners, precision="f32", method=method,
                    level_table=table)
    want = sample_filtered(dense, c, align_corners, address)
    np.testing.assert_allclose(got.cpu().numpy(), want, rtol=1e-5, atol=1e-6)
    empty = ic.sample(fp, dec, T(np.zeros((0, dim), np.float32)), mip, extent, precision="f32", method=method, level_table=table)
    assert tuple(empty.shape) == (0, 3)
    configure()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f32", "f16", "auto"])
def test_sample_at_texel_centres_is_decode_points(precision):
    """f = 0 on every axis: the sample is the texel's decode, bit for bit (pins the tap, PE and LOD mapping)."""
    ic = nic().image_compression
    rng = np.random.default_rng(340)
    for kind, align_corners in (("2d_mip0", False), ("2d_mip0", True), ("3d_m3", True)):
        fp, dec, table, method, mip, extent, _ = setup(kind)
        dim = 2 if method == 1 else 3
        s = extent if not (align_corners and method == 1) else 33      # S - 1 a power of two
        q = rng.integers(0, s, (2000, dim))
        c = ((q + 0.5) / s if not align_corners else q / (s - 1)).astype(np.float32)
        for dt in (torch.float32, torch.uint8):
            got = ic.sample(fp, dec, T(c), mip, size=s, align_corners=align_corners, precision=precision, out_dtype=dt,
                            method=method, level_table=table)
            want = ic.decode_points(fp, dec, torch.tensor(q), mip, precision=precision, out_dtype=dt, method=method,
                                    level_table=table)
            assert torch.equal(got, want), (kind, align_corners, dt)
    configure()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f16", "bf16"])
def test_tensor_core_sample_accuracy(precision):
    """North-star tolerance: 8-bit outputs within +-1 LSB of the fp32 sample for >= 99.9 %, PSNR against a target within
    0.05 dB."""
    ic = nic().image_compression
    size = 256
    configure(IMAGE_SIZE=size)
    fp = [T(g) for g in I.make_grids(size, 2, seed=350, no_mip=True, quantized=True)]
    dec = make_decoder(I.make_mlp(73, seed=351, gain=2.0))
    rng = np.random.default_rng(352)
    c = rng.random((131072, 2), dtype=np.float32)
    ref = ic.sample(fp, dec, T(c), 0, precision="f32", out_dtype=torch.uint8).cpu().numpy()
    got = ic.sample(fp, dec, T(c), 0, precision=precision, out_dtype=torch.uint8).cpu().numpy()
    within1, same, worst = lsb_stats(got, ref)
    assert within1 >= 0.999, (within1, same, worst)
    img = I.make_image(size, 2, seed=353)                                  # [3, S, S] with S the x axis first
    target = np.floor(sample_filtered(np.moveaxis(img, 0, -1), c, False) * 255 + 0.5)
    assert abs(psnr256(got, target) - psnr256(ref, target)) <= 0.05
    configure()


@pytest.mark.gpu
def test_fused_epilogue_equals_the_unfused_composition():
    """The tensor-core sample (fp32 out) against sum_k w_k * decode_points(tap_k) of the same kernel: only the summation
    order differs."""
    n = nic()
    ic, fp_def, L = n.image_compression, n.fp_def, n._lib
    rng = np.random.default_rng(360)
    for kind, precision in (("2d_mip0", "f16"), ("2d_mip3", "bf16"), ("3d_m3", "f16"), ("3d_m4", "bf16")):
        fp, dec, table, method, mip, extent, _ = setup(kind)
        dim = 2 if method == 1 else 3
        c = query_coords(rng, 4099, dim)
        for align_corners, address in ((False, "clamp"), (True, "wrap")):
            taps, w = tap_rule(c, (extent,) * dim, align_corners, address)
            got = ic.sample(fp, dec, T(c), mip, extent, address=address, align_corners=align_corners, precision=precision,
                            method=method, level_table=table).cpu().numpy()
            vals = ic.decode_points(fp, dec, torch.tensor(taps.reshape(-1, dim)), mip, precision=precision, method=method,
                                    level_table=table).cpu().numpy().reshape(taps.shape[0], taps.shape[1], -1)
            want = (w[..., None].astype(np.float64) * vals).sum(1)
            np.testing.assert_allclose(got, want, rtol=0, atol=1e-6)
    # from codes: decode_points_codes would take the code-resident kernel for this LUT; the sampler never does
    fp, dec, table, method, mip, extent, _ = setup("3d_m3")
    codes = fp_def.fp_savable(fp, 8)
    c = query_coords(rng, 4099, 3)
    taps, w = tap_rule(c, (extent,) * 3, True, "clamp")
    got = ic.sample_codes(codes, dec, T(c), 8, mip, extent, align_corners=True, method=method, level_table=table).cpu().numpy()
    L.set_option(dev(), L.OPT_DISABLE_FAST2D, 1)
    try:
        vals = ic.decode_points_codes(codes, dec, torch.tensor(taps.reshape(-1, 3)), 8, mip, out_dtype=torch.float32,
                                      method=method, level_table=table).cpu().numpy().reshape(taps.shape[0], 8, -1)
    finally:
        L.set_option(dev(), L.OPT_DISABLE_FAST2D, 0)
    np.testing.assert_allclose(got, (w[..., None].astype(np.float64) * vals).sum(1), rtol=0, atol=1e-6)
    configure()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f16", "bf16"])
@pytest.mark.parametrize("bits", [8, 4])
def test_sample_codes_equals_sample_of_loaded_grids(precision, bits):
    n = nic()
    ic, fp_def = n.image_compression, n.fp_def
    rng = np.random.default_rng(370 + bits)
    for kind in ("2d_mip0", "3d_m3"):
        fp, dec, table, method, mip, extent, _ = setup(kind)
        dim = 2 if method == 1 else 3
        codes = fp_def.fp_savable(fp, bits)
        loaded = fp_def.fp_load(codes, bits)
        c = T(query_coords(rng, 5000, dim))
        for dt in (torch.uint8, torch.float32):
            a = ic.sample_codes(codes, dec, c, bits, mip, extent, align_corners=True, precision=precision, out_dtype=dt, method=method,
                                level_table=table)
            b = ic.sample(loaded, dec, c, mip, extent, align_corners=True, precision=precision, out_dtype=dt, method=method,
                          level_table=table)
            assert torch.equal(a, b), (kind, dt)
    configure()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f32", "f16"])
def test_fractional_lod_blends_two_mips(precision):
    ic = nic().image_compression
    size = 64
    configure(IMAGE_SIZE=size, TF_NO_MIP=False, MAX_MIP_LEVEL=6)
    fp = [T(g) for g in I.make_grids(size, 2, seed=380, quantized=True)]
    dec = make_decoder(I.make_mlp(73, seed=381, gain=2.0))
    c = T(query_coords(np.random.default_rng(382), 3001, 2))
    for lod, m, t in ((1.25, 1, 0.25), (2.5, 2, 0.5), (0.75, 0, 0.75)):
        got = ic.sample(fp, dec, c, lod, precision=precision).cpu().numpy()
        a = ic.sample(fp, dec, c, m, precision=precision).cpu().numpy()
        b = ic.sample(fp, dec, c, m + 1, precision=precision).cpu().numpy()
        np.testing.assert_allclose(got, blend_lod(a, b, t), rtol=0, atol=1e-6)
    # the last mip of the table and a lod beyond MAX_MIP_LEVEL: one pass at the last mip
    last = ic.sample(fp, dec, c, 6, precision=precision)
    assert torch.equal(ic.sample(fp, dec, c, 7.5, precision=precision), last)
    assert torch.equal(ic.sample(fp, dec, c, -1.0, precision=precision), ic.sample(fp, dec, c, 0, precision=precision))
    configure()


@pytest.mark.gpu
def test_session_sample_reuses_the_tables():
    n = nic()
    ic = n.image_compression
    fp, dec, table, method, mip, extent, _ = setup("2d_mip0")
    c = T(query_coords(np.random.default_rng(390), 2048, 2))
    sess = ic.DecodeSession(fp, dec, precision="f16")
    first = sess.sample(c, 0, method=method, level_table=table)
    before = n.launch_count(dev())
    second = sess.sample(c, 0, method=method, level_table=table)
    assert n.launch_count(dev()) - before == 1
    assert torch.equal(first, second)
    assert torch.equal(first, ic.sample(fp, dec, c, 0, precision="f16", out_dtype=torch.uint8, method=method,
                                        level_table=table))
    configure()


@pytest.mark.gpu
def test_sample_errors():
    n = nic()
    ic, fp_def, L = n.image_compression, n.fp_def, n._lib
    fp, dec, table, method, mip, extent, _ = setup("2d_mip0")
    c = T(query_coords(np.random.default_rng(395), 64, 2))
    with pytest.raises(n.NicError) as e:                                   # texel 64 at step 1/4 reaches node 17 of 17
        ic.sample(fp, dec, c, 0, size=65, precision="f32", level_table=table)
    assert e.value.status == -4
    with pytest.raises(n.NicError) as e:
        ic.sample(fp, dec, c, 0, size=(64, 80), precision="f16", level_table=table)
    assert e.value.status == -4
    with pytest.raises(n.NicError) as e:
        ic.sample_codes(fp_def.fp_savable(fp, 8), dec, c, 8, 0, precision="f32", level_table=table)
    assert e.value.status == L.ERR_UNSUPPORTED
    with pytest.raises(n.NicError):
        ic.sample(fp, dec, c.cpu(), 0, level_table=table)
    with pytest.raises(n.NicError):
        ic.sample([g.cpu() for g in fp], dec, c, 0, level_table=table)
    with pytest.raises(TypeError):
        ic.sample(fp, dec, c.to(torch.int64), 0, level_table=table)
    with pytest.raises(TypeError):
        ic.sample(fp, dec, c.T.contiguous().T, 0, level_table=table)
    with pytest.raises(ValueError):
        ic.sample(fp, dec, c, 0, address="mirror", level_table=table)
    # the C ABI's own argument checks
    h = L.handle(dev())
    geom = L.make_geom(1, fp[0], fp[1], 1, 64, -2, 0, 6, L.PE_TRIANGULAR)
    m = L.make_mlp([p.detach().contiguous() for p in dec.parameters_list()])
    out = torch.empty((64, 3), device=dev())
    for address, ext in ((2, 64), (0, 0)):
        smp = L.NicSampler()
        smp.address, smp.extent[0], smp.extent[1], smp.extent[2] = address, ext, ext, 1
        rc = L.load_library().nic_sample(h, ctypes.byref(geom), L.ptr(fp[0]), L.ptr(fp[1]), L.ptr(c), ctypes.byref(smp),
                                         ctypes.byref(m), L.ptr(out), L.DT_F32, L.PREC_F32, L.stream_ptr(dev()))
        assert rc == -1, (address, ext)
    configure()
