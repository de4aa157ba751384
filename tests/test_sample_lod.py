"""Per-query level of detail (nic_sample_lod / nic_sample_lod_codes, image_compression.sample with a tensor lod or grad=):
the LOD oracle against a float64 loop, the ABI of NicMipChain and the host checks; on the GPU the fp32 arm against the
oracle and, bit for bit, against composed scalar samples, the derivative form, the tensor-core arm against the fp32 arm,
decode-from-codes, table reuse and the error cases."""
import ctypes
import math
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

import inputs as I
from helpers import T, configure, dev, lsb_stats, make_decoder, psnr256
from sample_lod_oracle import blend_mips, lod_from_derivatives, mip_pair, sample_lod

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32


def nic():
    import neural_image_compression_v2_b200 as n
    return n


def special_lods(rng, q, last):
    """lambda uniform in [-1, last + 1.5) with NaN, +-inf, negatives, exact integers and values beyond L among them."""
    lam = (rng.random(q, dtype=F32) * F32(last + 2.5) - F32(1)).astype(F32)
    lam[:8] = [np.nan, -np.inf, np.inf, -0.5, 0.0, 1.0, float(last), last + 3.0]
    return lam


# ------------------------------------------------------------------------------------------------ no GPU
def _loop_reference(frames, coords, lam):
    """Float64 loop: clamp, mip pair and a per-query bilinear sum with clamp addressing (align_corners False)."""
    last = len(frames) - 1
    out = np.zeros((coords.shape[0], frames[0].shape[-1]))
    for q in range(coords.shape[0]):
        lc = 0.0 if math.isnan(lam[q]) else min(max(float(lam[q]), 0.0), float(last))
        m = int(math.floor(lc))
        t = lc - m
        acc = []
        for mip in (m, min(m + 1, last)):
            f = frames[mip]
            v = np.zeros(f.shape[-1])
            axes = []
            for a in range(2):
                s = f.shape[a]
                p = min(max(float(coords[q, a]) * s - 0.5, -2.0 ** 24), 2.0 ** 24)
                i0 = math.floor(p)
                axes.append([(min(max(i0, 0), s - 1), 1 - (p - i0)), (min(max(i0 + 1, 0), s - 1), p - i0)])
            for ix, wx in axes[0]:
                for iy, wy in axes[1]:
                    v += wx * wy * f[ix, iy]
            acc.append(v)
        out[q] = (1 - t) * acc[0] + t * acc[1]
    return out


@pytest.mark.parametrize("constant", [False, True])
def test_lod_oracle_equals_a_float64_loop(constant):
    rng = np.random.default_rng(500 + constant)
    frames = [rng.random((16 >> i, 16 >> i, 3)) for i in range(5)]             # mips 0 .. 4, the last one texel
    coords = (rng.random((400, 2), dtype=F32) * F32(1.4) - F32(0.2)).astype(F32)
    lam = np.full(400, F32(2.375)) if constant else special_lods(rng, 400, 4)
    np.testing.assert_allclose(sample_lod(frames, coords, lam, False), _loop_reference(frames, coords, lam), rtol=0, atol=1e-6)


def test_lod_from_derivatives_edge_cases():
    """Zero derivatives give -inf (clamped to mip 0), the longer of the two screen axes wins, x is summed first."""
    ddx = np.array([[0, 0], [1 / 64, 0], [0, 1 / 16], [1 / 256, 0], [3.0, 4.0]], F32)
    ddy = np.array([[0, 0], [0, 1 / 128], [0, 0], [0, 1 / 512], [0, 0]], F32)
    lam = lod_from_derivatives(ddx, ddy, (64, 64))
    assert lam[0] == -np.inf
    np.testing.assert_allclose(lam[1:], [0.0, 2.0, -2.0, np.log2(5 * 64)], rtol=0, atol=1e-6)
    m, m1, t = mip_pair(np.array([np.nan, -np.inf, -1, 0, 2.5, 6, 7.25], F32), 6)
    assert m.tolist() == [0, 0, 0, 0, 2, 6, 6] and m1.tolist() == [1, 1, 1, 1, 3, 6, 6]
    assert t.tolist() == [0, 0, 0, 0, 0.5, 0, 0]
    # at t = 0 the blend is S_m exactly, whatever S_m1 is
    a = np.array([[0.1, 0.7]], F32)
    assert np.array_equal(blend_mips(a, np.array([[0.9, 0.3]], F32), np.zeros(1, F32)), a)


def test_mip_chain_struct_layout_matches_the_binding(tmp_path):
    L = nic()._lib
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "nic.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(NicMipChain));', '  printf("max %d\\n", NIC_MAX_MIPS);']
    for field, _ in L.NicMipChain._fields_:
        lines.append(f'  printf("{field} %zu\\n", offsetof(NicMipChain, {field}));')
    lines += ['  return 0;', '}']
    src = tmp_path / "chain.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "chain"
    subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split("\n")
    got = {l.split()[0]: int(l.split()[1]) for l in out if l.strip()}
    assert got["size"] == ctypes.sizeof(L.NicMipChain)
    assert got["max"] == L.MAX_MIPS
    for field, _ in L.NicMipChain._fields_:
        assert got[field] == getattr(L.NicMipChain, field).offset, field


def test_host_checks_of_the_lod_inputs():
    """dtype, shape and device of lod / ddx / ddy, lod together with grad, and size with a per-query lod are refused before
    anything is launched."""
    n = nic()
    ic = n.image_compression
    configure()
    dec = ic.ColorDecoder(in_channels=73, hidden=64, out_channels=3)
    fp = [torch.zeros(12, 129, 129), torch.zeros(12, 65, 65)]
    c = torch.zeros((4, 2), dtype=torch.float32)
    lod = torch.zeros(4, dtype=torch.float32)
    d = torch.zeros((4, 2), dtype=torch.float32)
    with pytest.raises(TypeError):
        ic.sample(fp, dec, c, lod.to(torch.float64))
    with pytest.raises(TypeError):
        ic.sample(fp, dec, c, torch.zeros((2, 4), dtype=torch.float32).T[0])
    with pytest.raises(ValueError):
        ic.sample(fp, dec, c, torch.zeros(5, dtype=torch.float32))
    with pytest.raises(ValueError):
        ic.sample(fp, dec, c, torch.zeros((4, 1), dtype=torch.float32))
    with pytest.raises(n.NicError):                                       # a host lod: no CPU fallback
        ic.sample(fp, dec, c, lod)
    with pytest.raises(TypeError):
        ic.sample(fp, dec, c, grad=(d, d.to(torch.float16)))
    with pytest.raises(ValueError):
        ic.sample(fp, dec, c, grad=(d, torch.zeros((4, 3), dtype=torch.float32)))
    with pytest.raises(TypeError):
        ic.sample(fp, dec, c, grad=d)
    with pytest.raises(n.NicError):
        ic.sample(fp, dec, c, grad=(d, d))
    with pytest.raises(ValueError):
        ic.sample(fp, dec, c, lod, grad=(d, d))
    with pytest.raises(ValueError):
        ic.sample(fp, dec, c, lod, size=64)
    with pytest.raises(ValueError):
        ic.sample(fp, dec, c, grad=(d, d), size=64)
    with pytest.raises(ValueError):
        ic.sample_codes([g.to(torch.uint8) for g in fp], dec, c, 8, lod, size=64)


# ------------------------------------------------------------------------------------------------ GPU
def query_coords(rng, q, dim):
    """Random coordinates in [-0.25, 1.25) with 0, 1, points outside [0, 1] and NaN among them."""
    c = (rng.random((q, dim), dtype=F32) * F32(1.5) - F32(0.25)).astype(F32)
    c[:6] = [[0.0] * dim, [1.0] * dim, [-0.3] * dim, [1.7] * dim, [np.nan] * dim, [0.5] * dim]
    c[6, 0] = np.nan
    return c


_MODELS = {}


def model(kind):
    """(grids, params, table, method, size, last, frames) of a test model with mips; frames are the oracle's decoded mips.
    2-D: 64^2, mips 0 .. 6 (mips 0-3 on pyramid level 0, 4-6 on level 1; mip 3 at step 2 without G1 interpolation, mip 6 one
    texel).  3-D: 32^3, mips 0 .. 5 on two pyramid levels (mip 3 at step 2, mip 5 one texel)."""
    if kind in _MODELS:
        return _MODELS[kind]
    from oracle import nic_oracle as O
    if kind == "2d":
        method, size, dim, seed = 1, 64, 2, 520
    else:
        method, size, dim, seed = (3, 32, 3, 530) if kind == "3d_m3" else (4, 32, 3, 540)
    grids = I.make_grids(size, dim, seed=seed, quantized=True)
    cin = 73 if method == 1 else (127 if method == 3 else 79)
    params = I.make_mlp(cin, seed=seed + 1, gain=2.0)
    table = O.create_pyramid_mip_levels(size, size // 4)
    last = int(math.log2(size))
    frames = [O.decode_block(grids, params, size >> mip, mip, table, method, use_tri_pe=True) for mip in range(last + 1)]
    _MODELS[kind] = (grids, params, table, method, size, last, frames)
    return _MODELS[kind]


def setup(kind):
    grids, params, table, method, size, last, frames = model(kind)
    if method == 1:
        configure(IMAGE_SIZE=size, TF_NO_MIP=False, MAX_MIP_LEVEL=last)
    else:
        configure(IMAGE_SIZE=size, IMAGE_DIMENSION=3, COMPRESSION_METHOD=method, TF_NO_MIP=False, MAX_MIP_LEVEL=last)
    return [T(g) for g in grids], make_decoder(params), table, method, last, frames


def _sample(ic, fp, dec, c, lod, method, table, **kw):
    return ic.sample(fp, dec, c, lod, method=method, level_table=table, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["2d", "3d_m3", "3d_m4"])
@pytest.mark.parametrize("address", ["clamp", "wrap"])
@pytest.mark.parametrize("align_corners", [False, True])
def test_f32_lod_sample_equals_oracle(kind, address, align_corners):
    ic = nic().image_compression
    fp, dec, table, method, last, frames = setup(kind)
    dim = 2 if method == 1 else 3
    rng = np.random.default_rng(550)
    c = query_coords(rng, 1003, dim)                                      # not a multiple of 32
    lam = special_lods(rng, 1003, last)
    got = _sample(ic, fp, dec, T(c), T(lam), method, table, address=address, align_corners=align_corners, precision="f32")
    want = sample_lod(frames, c, lam, align_corners, address)
    np.testing.assert_allclose(got.cpu().numpy(), want, rtol=1e-5, atol=1e-6)
    empty = _sample(ic, fp, dec, T(np.zeros((0, dim), F32)), T(np.zeros(0, F32)), method, table, precision="f32")
    assert tuple(empty.shape) == (0, 3)
    configure()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["2d", "3d_m4"])
def test_f32_lod_sample_is_the_composition_of_scalar_samples(kind):
    """lambda = k / 64 (t exact in both paths): the fp32 arm equals, bit for bit, scalar samples at every mip blended with
    nic.h's fp32 sequence; a constant lambda tensor equals the scalar sample at that lod."""
    ic = nic().image_compression
    fp, dec, table, method, last, _ = setup(kind)
    dim = 2 if method == 1 else 3
    rng = np.random.default_rng(560)
    c = T(query_coords(rng, 2011, dim))
    lam = (rng.integers(-64, 64 * (last + 2), 2011) / 64).astype(F32)
    lam[:3] = [0, last, last + 1]
    per_mip = [_sample(ic, fp, dec, c, i, method, table, precision="f32").cpu().numpy() for i in range(last + 1)]
    m, m1, t = mip_pair(lam, last)
    q = np.arange(len(lam))
    want = blend_mips(np.stack(per_mip)[m, q], np.stack(per_mip)[m1, q], t)
    got = _sample(ic, fp, dec, c, T(lam), method, table, precision="f32").cpu().numpy()
    assert np.array_equal(got, want)
    got8 = _sample(ic, fp, dec, c, T(lam), method, table, precision="f32", out_dtype=torch.uint8).cpu().numpy()
    want8 = np.clip(np.floor((want * F32(255)).astype(F32) + F32(0.5)), 0, 255).astype(np.uint8)
    assert np.array_equal(got8, want8)
    for lod in (1.25, 2.5, 3.0, last - 0.75):
        for dt in (torch.float32, torch.uint8):
            const = T(np.full(2011, lod, F32))
            assert torch.equal(_sample(ic, fp, dec, c, const, method, table, precision="f32", out_dtype=dt),
                               _sample(ic, fp, dec, c, lod, method, table, precision="f32", out_dtype=dt)), (lod, dt)
    configure()


def perspective_derivatives(rng, q, dim, size):
    """Derivatives whose lambda spans [-3, L + 3]: the longer axis scaled from 1/8 to 8 x the mip-chain's range."""
    scale = (2.0 ** rng.uniform(-3, math.log2(size) + 3, q)).astype(F32) / F32(size)
    ddx = (rng.normal(size=(q, dim)).astype(F32) * scale[:, None]).astype(F32)
    ddy = (rng.normal(size=(q, dim)).astype(F32) * scale[:, None] * F32(0.5)).astype(F32)
    ddx[:2] = 0
    ddy[:2] = 0
    return ddx, ddy


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["2d", "3d_m3"])
def test_derivative_form_equals_the_lod_form(kind):
    ic = nic().image_compression
    fp, dec, table, method, last, _ = setup(kind)
    dim = 2 if method == 1 else 3
    size = 64 if method == 1 else 32
    rng = np.random.default_rng(570)
    c = T(query_coords(rng, 3001, dim))
    ddx, ddy = perspective_derivatives(rng, 3001, dim, size)
    lam = lod_from_derivatives(ddx, ddy, (size,) * dim)
    assert (lam < 0).any() and (lam > last).any() and np.isneginf(lam[:2]).all()
    got = _sample(ic, fp, dec, c, None, method, table, precision="f32", grad=(T(ddx), T(ddy)))
    want = _sample(ic, fp, dec, c, T(lam), method, table, precision="f32")
    np.testing.assert_allclose(got.cpu().numpy(), want.cpu().numpy(), rtol=0, atol=1e-5)
    configure()


def smooth_target(c):
    """A smooth 8-bit reference signal at the query coordinates (only its distance to the two arms matters)."""
    c = np.nan_to_num(np.asarray(c, np.float64))
    v = 0.5 + 0.4 * np.sin(5 * c[:, :1]) * np.cos(3 * c[:, 1:2])
    return np.floor(np.repeat(v, 3, 1) * 255 + 0.5)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f16", "bf16"])
@pytest.mark.parametrize("kind", ["2d", "3d_m3", "3d_m4"])
def test_tensor_core_lod_sample_accuracy(precision, kind):
    """The bar of test_sample.py: 8-bit outputs within +-1 LSB of the fp32 arm for >= 99.9 %, PSNR within 0.05 dB."""
    ic = nic().image_compression
    fp, dec, table, method, last, _ = setup(kind)
    dim = 2 if method == 1 else 3
    size = 64 if method == 1 else 32
    rng = np.random.default_rng(580)
    q = 65536 if dim == 2 else 16384
    c = rng.random((q, dim), dtype=F32)
    lam = (rng.random(q, dtype=F32) * F32(last + 1) - F32(0.5)).astype(F32)
    ddx, ddy = perspective_derivatives(rng, q, dim, size)
    for lod, grad in ((T(lam), None), (None, (T(ddx), T(ddy)))):
        ref = _sample(ic, fp, dec, T(c), lod, method, table, precision="f32", out_dtype=torch.uint8, grad=grad).cpu().numpy()
        got = _sample(ic, fp, dec, T(c), lod, method, table, precision=precision, out_dtype=torch.uint8,
                      grad=grad).cpu().numpy()
        within1, same, worst = lsb_stats(got, ref)
        assert within1 >= 0.999, (within1, same, worst)
        target = smooth_target(c)
        assert abs(psnr256(got, target) - psnr256(ref, target)) <= 0.05
    configure()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f16", "bf16"])
@pytest.mark.parametrize("bits", [8, 4])
def test_lod_sample_codes_equals_sample_of_loaded_grids(precision, bits):
    n = nic()
    ic, fp_def = n.image_compression, n.fp_def
    rng = np.random.default_rng(590 + bits)
    for kind in ("2d", "3d_m3"):
        fp, dec, table, method, last, _ = setup(kind)
        dim = 2 if method == 1 else 3
        codes = fp_def.fp_savable(fp, bits)
        loaded = fp_def.fp_load(codes, bits)
        c = T(query_coords(rng, 5000, dim))
        lam = T(special_lods(rng, 5000, last))
        for dt in (torch.uint8, torch.float32):
            a = ic.sample_codes(codes, dec, c, bits, lam, align_corners=True, precision=precision, out_dtype=dt, method=method,
                                level_table=table)
            b = ic.sample(loaded, dec, c, lam, align_corners=True, precision=precision, out_dtype=dt, method=method,
                          level_table=table)
            assert torch.equal(a, b), (kind, dt)
    configure()


@pytest.mark.gpu
def test_session_lod_sample_reuses_the_chain_tables():
    n = nic()
    ic = n.image_compression
    fp, dec, table, method, last, _ = setup("2d")
    rng = np.random.default_rng(600)
    c = T(query_coords(rng, 2048, 2))
    lam = T(special_lods(rng, 2048, last))
    sess = ic.DecodeSession(fp, dec, precision="f16")
    first = sess.sample(c, lam, method=method, level_table=table)
    before = n.launch_count(dev())
    second = sess.sample(c, lam, method=method, level_table=table)
    assert n.launch_count(dev()) - before == 1
    assert torch.equal(first, second)
    sess.refresh()
    before = n.launch_count(dev())
    third = sess.sample(c, lam, method=method, level_table=table)
    assert n.launch_count(dev()) - before > 1
    assert torch.equal(first, third)
    assert torch.equal(first, ic.sample(fp, dec, c, lam, precision="f16", out_dtype=torch.uint8, method=method,
                                        level_table=table))
    configure()


@pytest.mark.gpu
def test_lod_sample_errors():
    n = nic()
    ic, fp_def, L = n.image_compression, n.fp_def, n._lib
    fp, dec, table, method, last, _ = setup("2d")
    rng = np.random.default_rng(610)
    c = T(query_coords(rng, 64, 2))
    lam = T(special_lods(rng, 64, last))
    d = T(np.zeros((64, 2), F32))
    with pytest.raises(n.NicError) as e:
        ic.sample_codes(fp_def.fp_savable(fp, 8), dec, c, 8, lam, precision="f32", level_table=table)
    assert e.value.status == L.ERR_UNSUPPORTED
    # the C ABI's own argument checks
    h = L.handle(dev())
    m = L.make_mlp([p.detach().contiguous() for p in dec.parameters_list()])
    out = torch.empty((64, 3), device=dev())

    def call(chain, lod, ddx, ddy):
        return L.load_library().nic_sample_lod(h, ctypes.byref(chain), L.ptr(c), L.ptr(lod), L.ptr(ddx), L.ptr(ddy),
                                               ctypes.byref(m), L.ptr(out), L.DT_F32, L.PREC_F32, L.stream_ptr(dev()))

    chain, _ = ic._mip_chain(fp, 64, "clamp", False, method, table)
    assert call(chain, lam, None, None) == 0
    assert call(chain, None, d, d) == 0
    for lod, ddx, ddy in ((lam, d, d), (lam, d, None), (None, None, None), (None, d, None)):
        assert call(chain, lod, ddx, ddy) == -1
    for num in (0, 17):
        bad, _ = ic._mip_chain(fp, 64, "clamp", False, method, table)
        bad.num_mips = num
        assert call(bad, lam, None, None) == -1, num
    bad, _ = ic._mip_chain(fp, 64, "clamp", False, method, table)
    bad.extent[0][0] = 65                                                 # texel 64 at step 1/4 reaches node 17 of 17
    assert call(bad, lam, None, None) == -4
    bad, _ = ic._mip_chain(fp, 64, "clamp", False, method, table)
    bad.geom[2].method = 3                                                # mips disagree on the method
    assert call(bad, lam, None, None) == -1
    configure()
