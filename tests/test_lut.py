"""Applying a baked 3-D colour LUT (nic_lut_pack / nic_lut_apply, image_compression.bake_lut* / BakedLut): the oracle of
the two interpolations against float64 restatements, the ABI of NicLut and the host checks; on the GPU the fp32 arm against
the oracle bit for bit, trilinear against `sample`, the tensor-core bake's accuracy, baking from codes, the neutral axis,
shapes and alignment, and the C error codes."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

import inputs as I
from helpers import T, configure, dev, lsb_stats, make_decoder, psnr256
from lut_oracle import apply as oracle_apply
from lut_oracle import tetrahedral, to_u8, trilinear, unit_coords
from sample_oracle import sample_filtered

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32


def nic():
    import neural_image_compression_v2_b200 as n
    return n


def special_coords(rng, q):
    """float32 coordinates in [-0.25, 1.25) with 0, 1, ties, out-of-range values, NaN and +-inf among them."""
    c = (rng.random((q, 3), dtype=np.float32) * F32(1.5) - F32(0.25)).astype(F32)
    c[:12] = [[0, 0, 0], [1, 1, 1], [0.5, 0.5, 0.5], [0.3, 0.3, 0.7], [0.7, 0.3, 0.3], [0.3, 0.7, 0.3], [-0.5, 0.2, 1.5],
              [np.nan, 0.5, 0.5], [0.5, np.inf, 0.5], [0.5, 0.5, -np.inf], [np.nan, np.nan, np.nan], [2.0, -1.0, 0.25]]
    return c


# ------------------------------------------------------------------------------------------------ no GPU
def tetra_six_cases(dense, u):
    """float64 restatement: the six tetrahedra of the unit cube written out case by case."""
    out = np.zeros((u.shape[0], dense.shape[3]))
    ext = dense.shape[:3]
    for q in range(u.shape[0]):
        lo, hi, f = [], [], []
        for a in range(3):
            p = float(u[q, a]) * (ext[a] - 1)
            p = -2.0 ** 24 if np.isnan(p) else min(max(p, -2.0 ** 24), 2.0 ** 24)
            i0 = np.floor(p)
            lo.append(int(min(max(i0, 0), ext[a] - 1)))
            hi.append(int(min(max(i0 + 1, 0), ext[a] - 1)))
            f.append(p - i0)
        fx, fy, fz = f

        def c(x, y, z):
            return dense[hi[0] if x else lo[0], hi[1] if y else lo[1], hi[2] if z else lo[2]].astype(np.float64)

        if fx >= fy >= fz:
            v = (1 - fx) * c(0, 0, 0) + (fx - fy) * c(1, 0, 0) + (fy - fz) * c(1, 1, 0) + fz * c(1, 1, 1)
        elif fx >= fz >= fy:
            v = (1 - fx) * c(0, 0, 0) + (fx - fz) * c(1, 0, 0) + (fz - fy) * c(1, 0, 1) + fy * c(1, 1, 1)
        elif fz >= fx >= fy:
            v = (1 - fz) * c(0, 0, 0) + (fz - fx) * c(0, 0, 1) + (fx - fy) * c(1, 0, 1) + fy * c(1, 1, 1)
        elif fy >= fx >= fz:
            v = (1 - fy) * c(0, 0, 0) + (fy - fx) * c(0, 1, 0) + (fx - fz) * c(1, 1, 0) + fz * c(1, 1, 1)
        elif fy >= fz >= fx:
            v = (1 - fy) * c(0, 0, 0) + (fy - fz) * c(0, 1, 0) + (fz - fx) * c(0, 1, 1) + fx * c(1, 1, 1)
        else:
            v = (1 - fz) * c(0, 0, 0) + (fz - fy) * c(0, 0, 1) + (fy - fx) * c(0, 1, 1) + fx * c(1, 1, 1)
        out[q] = v
    return out


def test_trilinear_oracle_equals_sample_filtered():
    rng = np.random.default_rng(500)
    dense = rng.random((9, 6, 11, 3)).astype(F32)
    u = special_coords(rng, 2000)
    got = trilinear(dense, u)
    assert got.dtype == np.float32
    np.testing.assert_allclose(got, sample_filtered(dense, u, True, "clamp"), rtol=0, atol=1e-6)
    img = rng.integers(0, 256, (777, 3), dtype=np.uint8)
    np.testing.assert_allclose(oracle_apply(dense, img, "trilinear"),
                               sample_filtered(dense, unit_coords(img), True, "clamp"), rtol=0, atol=1e-6)


def test_tetrahedral_oracle_equals_the_six_cases():
    rng = np.random.default_rng(510)
    dense = rng.random((7, 10, 5, 4)).astype(F32)
    u = special_coords(rng, 3000)
    u[12:400] = np.round(u[12:400] * 4) / 4                              # many ties between the fractions
    got = tetrahedral(dense, u)
    assert got.dtype == np.float32
    np.testing.assert_allclose(got, tetra_six_cases(dense, u), rtol=0, atol=1e-6)


@pytest.mark.parametrize("interpolation", ["trilinear", "tetrahedral"])
def test_affine_tables_are_reproduced(interpolation):
    rng = np.random.default_rng(520)
    ext = (17, 9, 33)
    A = rng.uniform(-0.3, 0.3, (3, 3))
    b = np.array([0.4, 0.5, 0.3])
    grid = np.stack(np.meshgrid(*[np.arange(s) / (s - 1) for s in ext], indexing="ij"), -1)     # [Sx, Sy, Sz, 3]
    dense = (grid @ A.T + b).astype(F32)
    u = rng.random((5000, 3), dtype=np.float32)
    got = oracle_apply(dense, u, interpolation)
    np.testing.assert_allclose(got, u.astype(np.float64) @ A.T + b, rtol=0, atol=1e-6)


def test_tetrahedral_equals_trilinear_on_edges_and_faces():
    """Where two of the three fractions are 0 both rules interpolate along one edge, bit for bit."""
    rng = np.random.default_rng(530)
    dense = rng.random((17, 17, 17, 3)).astype(F32)
    n = 3000
    u = (rng.integers(0, 17, (n, 3)) / 16).astype(F32)                   # texel centres: S - 1 = 16, exact
    axis = rng.integers(0, 3, n)
    u[np.arange(n), axis] = rng.random(n, dtype=np.float32)
    np.testing.assert_array_equal(tetrahedral(dense, u), trilinear(dense, u))


def test_lut_struct_layout_matches_the_binding(tmp_path):
    L = nic()._lib
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "nic.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(NicLut));']
    for field, _ in L.NicLut._fields_:
        lines.append(f'  printf("{field} %zu\\n", offsetof(NicLut, {field}));')
    lines += ['  printf("interp %d %d\\n", NIC_INTERP_TRILINEAR, NIC_INTERP_TETRAHEDRAL);', '  return 0;', '}']
    src = tmp_path / "lut.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "lut"
    subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split("\n")
    got = {l.split()[0]: l.split()[1:] for l in out if l.strip()}
    assert int(got["size"][0]) == ctypes.sizeof(L.NicLut)
    for field, _ in L.NicLut._fields_:
        assert int(got[field][0]) == getattr(L.NicLut, field).offset, field
    assert got["interp"] == [str(L.INTERP_TRILINEAR), str(L.INTERP_TETRAHEDRAL)]


def test_host_checks():
    """dtype, shape and device are checked before anything is launched; host tensors are refused (no CPU fallback)."""
    n = nic()
    ic = n.image_compression
    lut = ic.BakedLut(torch.zeros((2, 2, 2, 4)), (2, 2, 2), 3)
    img = torch.zeros((4, 3), dtype=torch.uint8)
    with pytest.raises(TypeError):
        lut.apply(img.to(torch.int64))
    with pytest.raises(TypeError):
        lut.apply(torch.zeros((3, 4), dtype=torch.uint8).T)
    with pytest.raises(TypeError):
        lut.apply([[0, 0, 0]])
    with pytest.raises(ValueError):
        lut.apply(torch.zeros((4, 4), dtype=torch.uint8))
    with pytest.raises(ValueError):
        lut.apply(img, interpolation="nearest")
    with pytest.raises(TypeError):
        lut.apply(img, out_dtype=torch.float16)
    with pytest.raises(n.NicError) as e:
        lut.apply(img)
    assert e.value.status == -3
    with pytest.raises(TypeError):
        ic.BakedLut.from_table(torch.zeros((2, 2, 2, 3), dtype=torch.float64))
    with pytest.raises(ValueError):
        ic.BakedLut.from_table(torch.zeros((2, 2, 2, 5)))
    with pytest.raises(ValueError):
        ic.BakedLut.from_table(torch.zeros((4, 4, 3)))
    with pytest.raises(TypeError):
        ic.BakedLut.from_table(torch.zeros((2, 2, 2, 3)), table_dtype=torch.bfloat16)
    with pytest.raises(n.NicError) as e:
        ic.BakedLut.from_table(torch.zeros((2, 2, 2, 3)))
    assert e.value.status == -3
    configure()
    dec = ic.ColorDecoder(in_channels=73, hidden=64, out_channels=3)
    with pytest.raises(ValueError):                                       # a 2-D model is a texture
        ic.bake_lut([torch.zeros(12, 129, 129), torch.zeros(12, 65, 65)], dec)
    with pytest.raises(ValueError):
        ic.bake_lut_codes([torch.zeros(12, 129, 129, dtype=torch.uint8)] * 2, dec, 8, method=1)


# ------------------------------------------------------------------------------------------------ GPU
_MODELS = {}


def lut_model(method):
    """The config-4 shape: a method-3 / method-4 model of a 64^3 volume whose grids hold one node more than the 64-texel
    mip needs (18^3 and 10^3), so a 65^3 LUT at step 1/4 stays inside them."""
    if method not in _MODELS:
        rng = np.random.default_rng(540 + method)
        lo, hi = I.q_range(8)
        grids = [np.floor(rng.uniform(lo, hi, (12, 18, 18, 18)) * 255 + 0.5).astype(F32) / F32(255),
                 np.floor(rng.uniform(lo, hi, (12, 10, 10, 10)) * 255 + 0.5).astype(F32) / F32(255)]
        _MODELS[method] = (grids, I.make_mlp(127 if method == 3 else 79, seed=541, gain=2.0))
    grids, params = _MODELS[method]
    configure(IMAGE_SIZE=64, IMAGE_DIMENSION=3, COMPRESSION_METHOD=method)
    return [T(g) for g in grids], make_decoder(params), {0: 0}


def all_colours():
    i = torch.arange(1 << 24, device=dev(), dtype=torch.int32)
    return torch.stack([i >> 16, (i >> 8) & 255, i & 255], 1).to(torch.uint8).contiguous()


@pytest.mark.gpu
@pytest.mark.parametrize("method", [3, 4])
def test_f32_apply_equals_oracle(method):
    ic = nic().image_compression
    fp, dec, table = lut_model(method)
    img = all_colours()
    for size in (65, (65, 33, 50)):
        lut = ic.bake_lut(fp, dec, 0, size=size, precision="f32", method=method, level_table=table)
        assert lut.table.dtype == torch.float32 and lut.cout == 3
        dense = lut.table[..., :3].cpu().numpy()
        assert not lut.table[..., 3].any()
        np.testing.assert_array_equal(dense, ic.decode(fp, dec, 0, size=size, precision="f32", method=method,
                                                       level_table=table).cpu().numpy())
        rng = np.random.default_rng(550)
        fimg = T(special_coords(rng, 100003))
        for interp in ("trilinear", "tetrahedral"):
            chunks = [img] if size == 65 else [img[::97].contiguous()]
            for src in chunks:
                got32 = lut.apply(src, interp, torch.float32).cpu().numpy()
                got8 = lut.apply(src, interp, torch.uint8).cpu().numpy()
                s = src.cpu().numpy()
                for k in range(0, s.shape[0], 1 << 20):                   # the oracle in chunks bounds host memory
                    want = oracle_apply(dense, s[k:k + (1 << 20)], interp)
                    np.testing.assert_array_equal(got32[k:k + (1 << 20)], want, err_msg=f"{size} {interp} u8 in")
                    np.testing.assert_array_equal(got8[k:k + (1 << 20)], to_u8(want), err_msg=f"{size} {interp} u8 out")
            want = oracle_apply(dense, fimg.cpu().numpy(), interp)
            np.testing.assert_array_equal(lut.apply(fimg, interp, torch.float32).cpu().numpy(), want, err_msg=f"{size} f32")
            np.testing.assert_array_equal(lut.apply(fimg, interp, torch.uint8).cpu().numpy(), to_u8(want))
    configure()


@pytest.mark.gpu
def test_f32_trilinear_equals_sample():
    ic = nic().image_compression
    fp, dec, table = lut_model(3)
    lut = ic.bake_lut(fp, dec, 0, size=65, precision="f32", level_table=table)
    host = np.random.default_rng(560).integers(0, 256, (200003, 3), dtype=np.uint8)
    img = T(host)
    coords = T(unit_coords(host))         # v / 255 correctly rounded (torch divides by a scalar through its reciprocal)
    for dt in (torch.float32, torch.uint8):
        want = ic.sample(fp, dec, coords, 0, size=65, align_corners=True, precision="f32", out_dtype=dt, level_table=table)
        assert torch.equal(lut.apply(img, "trilinear", dt), want), dt
    configure()


def smooth_image(h, w, seed):
    """A seeded smooth image plus noise, [h, w, 3] uint8: coherent like a photograph."""
    g = torch.Generator(device=dev()).manual_seed(seed)
    low = torch.rand((1, 3, h // 32 + 2, w // 32 + 2), generator=g, device=dev())
    img = torch.nn.functional.interpolate(low, size=(h, w), mode="bicubic", align_corners=False)[0].permute(1, 2, 0)
    img = img + 0.03 * torch.randn((h, w, 3), generator=g, device=dev())
    return torch.floor(img.clamp(0, 1) * 255 + 0.5).to(torch.uint8).contiguous()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f16", "bf16"])
def test_tensor_core_bake_accuracy(precision):
    n = nic()
    ic, fp_def = n.image_compression, n.fp_def
    fp, dec, table = lut_model(3)
    img = smooth_image(540, 960, 570)
    ref = ic.bake_lut(fp, dec, 0, size=65, precision="f32", level_table=table)
    lut = ic.bake_lut(fp, dec, 0, size=65, precision=precision, level_table=table)
    assert lut.table.dtype == torch.float16
    target = smooth_image(540, 960, 571).cpu().numpy()
    for interp in ("trilinear", "tetrahedral"):
        a = ref.apply(img, interp).cpu().numpy()
        b = lut.apply(img, interp).cpu().numpy()
        within1, same, worst = lsb_stats(b, a)
        assert within1 >= 0.999, (interp, within1, same, worst)
        assert abs(psnr256(b, target) - psnr256(a, target)) <= 0.05
    # the fp16 table alone: |delta| <= 2^-12 of a value in [0, 1], and the blend keeps it
    dense = ic.decode(fp, dec, 0, size=65, precision="f32", level_table=table)
    t32, t16 = ic.BakedLut.from_table(dense), ic.BakedLut.from_table(dense, torch.float16)
    for interp in ("trilinear", "tetrahedral"):
        d = (t16.apply(img, interp, torch.float32) - t32.apply(img, interp, torch.float32)).abs().max()
        assert float(d) <= 2.5e-4, (interp, float(d))
    # the fp16-table apply against today's product route on the same coordinates
    codes = fp_def.fp_savable(fp, 8)
    baked = ic.bake_lut_codes(codes, dec, 8, 0, size=65, precision=precision, level_table=table)
    flat = img.view(-1, 3)
    coords = T(unit_coords(flat.cpu().numpy()))
    want = ic.sample_codes(codes, dec, coords, 8, 0, size=65, align_corners=True, precision=precision, level_table=table)
    assert float((baked.apply(flat, "trilinear", torch.float32) - want).abs().max()) <= 3e-4
    want8 = ic.sample_codes(codes, dec, coords, 8, 0, size=65, align_corners=True, precision=precision,
                            out_dtype=torch.uint8, level_table=table)
    assert int((baked.apply(flat).to(torch.int32) - want8.to(torch.int32)).abs().max()) <= 1
    configure()


@pytest.mark.gpu
@pytest.mark.parametrize("method", [3, 4])
def test_bake_from_codes_equals_bake_of_loaded_grids(method):
    n = nic()
    ic, fp_def = n.image_compression, n.fp_def
    fp, dec, table = lut_model(method)
    codes = fp_def.fp_savable(fp, 8)
    a = ic.bake_lut_codes(codes, dec, 8, 0, size=65, level_table=table)
    b = ic.bake_lut(fp_def.fp_load(codes, 8), dec, 0, size=65, precision="f16", level_table=table)
    assert a.table.dtype == b.table.dtype == torch.float16 and a.extent == b.extent == (65, 65, 65)
    assert torch.equal(a.table, b.table)
    configure()


@pytest.mark.gpu
def test_tetrahedral_neutral_axis_is_the_diagonal_lerp():
    ic = nic().image_compression
    fp, dec, table = lut_model(4)
    lut = ic.bake_lut(fp, dec, 0, size=65, precision="f32", level_table=table)
    d = lut.table.cpu().numpy()
    v = np.arange(256, dtype=np.uint8)
    got = lut.apply(T(np.stack([v, v, v], 1)), "tetrahedral", torch.float32).cpu().numpy()
    p = (v.astype(F32) / F32(255) * F32(64)).astype(F32)
    i0 = np.floor(p)
    f = (p - i0).astype(F32)
    lo, hi = i0.astype(np.int64), np.minimum(i0.astype(np.int64) + 1, 64)
    want = (((F32(1) - f)[:, None] * d[lo, lo, lo, :3]).astype(F32) + (f[:, None] * d[hi, hi, hi, :3]).astype(F32)).astype(F32)
    np.testing.assert_array_equal(got, want)
    configure()


@pytest.mark.gpu
@pytest.mark.parametrize("cout", [1, 3, 4])
def test_shapes_alignment_and_empty_calls(cout):
    n = nic()
    ic = n.image_compression
    rng = np.random.default_rng(580 + cout)
    dense = T(rng.random((17, 12, 9, cout), dtype=np.float32))
    for table_dtype in (torch.float32, torch.float16):
        lut = ic.BakedLut.from_table(dense, table_dtype)
        assert lut.cout == cout and lut.extent == (17, 12, 9) and tuple(lut.table.shape) == (17, 12, 9, 4)
        for src_dtype in (torch.uint8, torch.float32):
            base = rng.integers(0, 256, (4099, 3), dtype=np.uint8)
            flat = T(base) if src_dtype == torch.uint8 else T(base.astype(F32) / F32(255) * F32(1.2) - F32(0.1))
            for interp in ("trilinear", "tetrahedral"):
                for dt in (torch.uint8, torch.float32):
                    ref = lut.apply(flat, interp, dt)
                    assert tuple(ref.shape) == (4099, cout) and ref.dtype == dt
                    want = oracle_apply(lut.table[..., :cout].float().cpu().numpy(), flat.cpu().numpy(), interp)
                    np.testing.assert_array_equal(ref.cpu().numpy(), to_u8(want) if dt == torch.uint8 else want)
                    for N in (0, 1, 15, 16, 17, 4097):
                        got = lut.apply(flat[:N].contiguous(), interp, dt)
                        assert tuple(got.shape) == (N, cout) and torch.equal(got, ref[:N]), N
                    assert torch.equal(lut.apply(flat[:4096].view(64, 64, 3), interp, dt), ref[:4096].view(64, 64, cout))
                    assert torch.equal(lut.apply(flat[:4096].view(4, 32, 32, 3), interp, dt),
                                       ref[:4096].view(4, 32, 32, cout))
                    # an input view one pixel into its buffer, an output view at an odd element offset
                    assert torch.equal(lut.apply(flat[1:], interp, dt), ref[1:])
                    buf = torch.empty(4098 * cout + 1, dtype=dt, device=dev())
                    view = buf[1:1 + 4098 * cout].view(4098, cout)
                    assert lut.apply(flat[1:], interp, dt, out=view) is view and torch.equal(view, ref[1:])
    lut = ic.BakedLut.from_table(dense)
    before = n.launch_count(dev())
    empty = lut.apply(torch.empty((0, 3), dtype=torch.uint8, device=dev()))
    assert tuple(empty.shape) == (0, cout) and n.launch_count(dev()) == before
    img = T(rng.integers(0, 256, (64, 3), dtype=np.uint8))
    with pytest.raises(ValueError):
        lut.apply(img, out=torch.empty((64, cout + 1), dtype=torch.uint8, device=dev()))
    with pytest.raises(ValueError):
        lut.apply(img, out=torch.empty((64, cout), dtype=torch.float32, device=dev()))
    buf = torch.empty(64 * 3 + 64 * cout, dtype=torch.uint8, device=dev())
    with pytest.raises(ValueError):                                       # not in place
        lut.apply(buf[:192].view(64, 3), out=buf[100:100 + 64 * cout].view(64, cout))
    with pytest.raises(n.NicError):
        lut.apply(img.cpu())


@pytest.mark.gpu
def test_lut_errors():
    n = nic()
    L = n._lib
    lib = L.load_library()
    h = L.handle(dev())
    st = L.stream_ptr(dev())
    table = torch.zeros((4, 4, 4, 4), device=dev())
    src = torch.zeros((64, 3), dtype=torch.uint8, device=dev())
    dst = torch.zeros((64, 3), dtype=torch.uint8, device=dev())

    def make(**kw):
        lut = L.NicLut()
        lut.table, lut.table_dtype, lut.cout = table.data_ptr(), L.DT_F32, 3
        for a in range(3):
            lut.extent[a] = 4
        for k, v in kw.items():
            if k == "extent":
                for a in range(3):
                    lut.extent[a] = v[a]
            else:
                setattr(lut, k, v)
        return lut

    def apply(lut, s=src, sd=L.DT_U8, pixels=64, d=dst, dd=L.DT_U8, interp=L.INTERP_TRILINEAR):
        return lib.nic_lut_apply(h, ctypes.byref(lut) if lut is not None else None, L.ptr(s), sd, pixels, L.ptr(d), dd,
                                 interp, st)

    assert apply(make()) == 0
    assert apply(make(), interp=L.INTERP_TETRAHEDRAL) == 0
    assert apply(None) == -1
    for kw in ({"table_dtype": L.DT_U8}, {"table_dtype": L.DT_BF16}, {"cout": 0}, {"cout": 5}, {"reserved": 1},
               {"extent": (4, 0, 4)}, {"table": None}):
        assert apply(make(**kw)) == -1, kw
    assert apply(make(), sd=L.DT_F16) == -1
    assert apply(make(), dd=L.DT_BF16) == -1
    assert apply(make(), interp=2) == -1
    assert apply(make(), pixels=-1) == -1
    assert apply(make(), s=None) == -1
    assert apply(make(), d=None) == -1
    assert apply(make(), d=src) == -1                                     # in place
    assert apply(make(), s=None, d=None, pixels=0) == 0
    assert apply(make(extent=(2048, 2048, 512))) == -2                   # 2^31 texels
    ext = (ctypes.c_int32 * 3)(4, 4, 4)
    dense = torch.zeros((4, 4, 4, 3), device=dev())
    pack = lib.nic_lut_pack
    assert pack(h, L.ptr(dense), ext, 3, L.ptr(table), L.DT_F32, st) == 0
    assert pack(h, L.ptr(dense), ext, 3, L.ptr(table), L.DT_U8, st) == -1
    assert pack(h, L.ptr(dense), ext, 5, L.ptr(table), L.DT_F32, st) == -1
    assert pack(h, None, ext, 3, L.ptr(table), L.DT_F32, st) == -1
    assert pack(h, L.ptr(dense), (ctypes.c_int32 * 3)(4, -1, 4), 3, L.ptr(table), L.DT_F32, st) == -1
    assert pack(h, L.ptr(dense), (ctypes.c_int32 * 3)(2048, 2048, 512), 3, L.ptr(table), L.DT_F32, st) == -2
    torch.cuda.synchronize()
