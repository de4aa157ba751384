"""The data front end of the training step (SURVEY §8(f) ranks 1, 3, 4): mip-pyramid builder, device-side crop sampler,
method-2 atlas, per-step metrics without host syncs.

CPU tests pin the oracle's restatement of Pillow's resample to outputs of the reference's own transform
(tests/golden/resize.npz, made by tests/golden/make_golden_data.py with torchvision + Pillow); GPU tests hold the kernels
to the same fixtures and to the oracle, bit for bit (integer / byte work)."""
import math
import os

import numpy as np
import pytest
import torch

import inputs as I
from helpers import T, configure, dev, load, make_decoder
from oracle import nic_oracle as O

RECT = ((23, 17), (61, 20), (30, 45), (80, 19), (7, 90))


# ------------------------------------------------------------------------------------------------ CPU: oracle vs fixtures
def test_oracle_pil_resize_matches_reference_transform():
    z = load("resize.npz")
    src = z["square_src"]
    for i in range(8):
        s = src.shape[0] >> i
        assert np.array_equal(O.pil_resize_bilinear(src, s, s), z[f"square_mip{i}"]), f"mip {i}"
    for h, w in RECT:
        assert np.array_equal(O.pil_resize_bilinear(z["rect_src"], h, w), z[f"rect_{h}x{w}"]), (h, w)
    t = O.to_tensor(z["square_mip2"])
    assert t.shape == (3, 32, 32) and t.dtype == np.float32 and t.max() <= 1.0


def test_oracle_sampler_and_atlas_properties():
    # origins stay inside the image and cover the whole range; the draw is a pure function of (seed, step, crop)
    o = O.random_crop_origins(5, 7, 4096, (64, 64), (16, 16))
    assert o.min() == 0 and o.max() == 48 and np.array_equal(o, O.random_crop_origins(5, 7, 4096, (64, 64), (16, 16)))
    assert not np.array_equal(o, O.random_crop_origins(5, 8, 4096, (64, 64), (16, 16)))
    counts = np.bincount(o[:, 0], minlength=49)
    assert counts.min() > 40 and counts.max() < 130            # uniform over 49 values, 4096 draws (mean 83.6)
    # Philox4x32-10 known-answer vector (Random123 kat_vectors: counter = key = 0)
    assert O.philox4x32_10(0, 0, 0) == (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)
    rng = np.random.default_rng(3)
    frames = rng.integers(0, 256, (10, 8, 8, 3)).astype(np.uint8)
    atlas = O.atlas_pack(frames, 32)
    assert atlas.shape == (32, 32, 3) and np.array_equal(O.atlas_unpack(atlas, 8, 10), frames)
    assert np.array_equal(atlas[8:16, 0:8], frames[4]) and not atlas[24:].any()


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_mip_pyramid_builder_bit_exact():
    """build_mip_pyramid == [ToTensor(Resize((S >> i, S >> i))(image)) for i] of the script (image_compression.py:433-442)."""
    import neural_image_compression_v2_b200 as n
    ic = n.image_compression
    z = load("resize.npz")
    src = T(z["square_src"])
    configure(IMAGE_SIZE=128, TF_NO_MIP=False, MAX_MIP_LEVEL=7)
    pyr = ic.build_mip_pyramid(src)
    assert len(pyr) == 8
    for i, p in enumerate(pyr):
        s = 128 >> i
        assert tuple(p.shape) == (3, s, s) and p.dtype == torch.float32
        assert np.array_equal(p.cpu().numpy(), O.to_tensor(z[f"square_mip{i}"])), f"mip {i}"
    rsrc = T(z["rect_src"])
    for h, w in RECT:
        f, u8 = ic.resize_image(rsrc, h, w, want_u8=True)
        assert np.array_equal(u8.cpu().numpy(), z[f"rect_{h}x{w}"]), (h, w)
        assert np.array_equal(f.cpu().numpy(), O.to_tensor(z[f"rect_{h}x{w}"]))
    # a frame of the benchmark size against the oracle on one channel-row band (the oracle is slow in Python)
    rng = np.random.default_rng(4)
    big = rng.integers(0, 256, (1024, 1024, 3)).astype(np.uint8)
    _, u8 = ic.resize_image(T(big), 64, 64, want_u8=True)
    assert np.array_equal(u8.cpu().numpy(), O.pil_resize_bilinear(big, 64, 64))


@pytest.mark.gpu
def test_device_side_sampler_matches_oracle():
    """nic_sample_crops_random: origins = the oracle's Philox draw, targets = the reference's per-crop slices (:42-47)."""
    import neural_image_compression_v2_b200 as n
    ic = n.image_compression
    rng = np.random.default_rng(11)
    for dim, size in ((2, 64), (3, 16)):
        imgs = [rng.random((3,) + (size >> m,) * dim).astype(np.float32) for m in range(3)]
        dimgs = [T(a) for a in imgs]
        for lod in range(3):
            for step in (0, 5):
                tg, coord = ic.random_crop_dataset_device(dimgs, 8, 6, lod, seed=1234, step=step, dim=dim)
                s = max(1, 8 // 2 ** lod)
                want = O.random_crop_origins(1234, step, 6, (size >> lod,) * dim, (s,) * dim)
                assert np.array_equal(coord.cpu().numpy(), want)
                assert np.array_equal(tg.cpu().numpy(), O.crop_targets(imgs[lod], want, s))


@pytest.mark.gpu
def test_atlas_round_trip():
    import neural_image_compression_v2_b200 as n
    ic = n.image_compression
    rng = np.random.default_rng(12)
    frames = rng.integers(0, 256, (16, 16, 16, 3)).astype(np.uint8)
    configure(IMAGE_SIZE=64, IMAGE_3D_SIZE=16, COMPRESSION_METHOD=2, IMAGE_DIMENSION=3)
    atlas = ic.flatten_movie_to_atlas(T(frames))
    assert np.array_equal(atlas.cpu().numpy(), O.atlas_pack(frames, 64))
    assert np.array_equal(ic.unflatten_atlas(atlas).cpu().numpy(), frames)
    odd = rng.integers(0, 256, (5, 8, 8, 1)).astype(np.uint8)          # fewer frames than tiles, one channel
    a2 = ic.flatten_movie_to_atlas(T(odd), image_size=28)
    assert np.array_equal(a2.cpu().numpy(), O.atlas_pack(odd, 28))
    assert np.array_equal(ic.unflatten_atlas(a2, 8, 5).cpu().numpy(), odd)
    with pytest.raises(n._lib.NicError):
        ic.flatten_movie_to_atlas(T(odd), image_size=16)               # 5 frames do not fit 2 x 2 tiles
    configure()


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["f32", "f16"])
def test_step_metrics_ring_matches_host_computation(prec):
    """flush_metrics(): per-step loss and the PSNR of the 8-bit-rounded outputs vs targets (image_compression.py:258-261,
    275-279) come back from the device ring in one copy and equal what the reference computes per step on the host."""
    import neural_image_compression_v2_b200 as n
    ic = n.image_compression
    size, crop, nc = 512, 256, 2
    configure(IMAGE_SIZE=size, NUM_EPOCHS=50)
    fp = [T(g) for g in I.make_grids(size, 2, seed=31, no_mip=True)]
    dec = make_decoder(I.make_mlp(73, seed=32))
    img = I.make_image(size, 2, seed=33)
    tr = ic.FusedTrainer(fp, dec, num_epochs=50, fp_bits=8, seed=2, precision=prec, metrics_ring=16)
    rng = np.random.default_rng(34)
    want, losses = [], []
    for s in range(40):                                  # 40 > ring of 16: exercises the ring roll-over
        coord = rng.integers(0, size - crop + 1, (nc, 2))
        tg = O.crop_targets(img, coord, crop)
        out = torch.empty((nc * crop * crop, 3), dtype=torch.float32, device=dev())
        losses.append(tr.step(T(coord), T(tg), 0, noise=False, out=out))
        o = out.cpu().numpy()
        t = tg.reshape(-1, 3)
        mse8 = float(np.mean((np.floor(o * np.float32(255) + np.float32(0.5)) - np.floor(t * np.float32(255) + np.float32(0.5))) ** 2))
        want.append((float(np.mean((o - t) ** 2, dtype=np.float64)), 10 * math.log10(65536.0 / mse8)))
        if s == 24:
            first = tr.flush_metrics()
            assert [m[0] for m in first] == list(range(25))
    rest = tr.flush_metrics()
    got = first + rest
    assert [m[0] for m in got] == list(range(40)) and tr.flush_metrics() == []
    for (step, loss, psnr), (wl, wp), handle in zip(got, want, losses):
        assert abs(loss - wl) <= 2e-5 * max(wl, 1e-6) + 1e-9, (step, loss, wl)
        assert abs(psnr - wp) <= 2e-3, (step, psnr, wp)
        assert float(handle) == loss                     # handles returned by step() stay valid across ring roll-overs


@pytest.mark.gpu
def test_step_sampled_trains_and_is_reproducible():
    """step_sampled = LOD draw + device sampler + fused step: two trainers with the same seed take identical steps
    (bit-identical parameters on the f32 path is too strict with float atomics; losses agree to rounding), the LOD
    sequence follows the reference's schedule, and the loss goes down."""
    import neural_image_compression_v2_b200 as n
    ic = n.image_compression
    size = 256
    configure(IMAGE_SIZE=size, TF_NO_MIP=False, MAX_MIP_LEVEL=8, NUM_EPOCHS=200, NUM_CROPS=4)
    img8 = np.floor(np.transpose(I.make_image(size, 2, seed=41), (1, 2, 0)) * 255 + 0.5).astype(np.uint8)
    pyr = ic.build_mip_pyramid(T(img8))
    runs = []
    for rep in range(2):
        fp = [T(g) for g in I.make_grids(size, 2, seed=42, no_mip=False)]
        dec = make_decoder(I.make_mlp(73, seed=43))
        tr = ic.FusedTrainer(fp, dec, num_epochs=200, fp_bits=8, seed=9, precision="f16")
        lods = [tr.step_sampled(pyr)[1] for _ in range(120)]
        runs.append((lods, [m[1] for m in tr.flush_metrics()]))
    assert runs[0][0] == runs[1][0]
    np.testing.assert_allclose(runs[0][1], runs[1][1], rtol=5e-2)
    lods, losses = runs[0]
    assert min(lods) == 0 and max(lods) >= 2 and lods.count(0) > 60          # P(lod = k) ~ 4^-k, uniform every 20th step
    assert np.mean(losses[-20:]) < 0.5 * np.mean(losses[:20])
    configure()


# ------------------------------------------------------------------------------------------------ host file helpers (f4)
def test_host_file_helpers_formats(tmp_path):
    """save_result_to_csv / make_filename_by_seq / readClip / timelaps (utils.py:37-113): file formats as the reference
    writes them — checked against the format spelled out here, and against the reference's own functions as well when
    NIC_REFERENCE_DIR names the reference's Projects/ directory.  No device involved."""
    import importlib.util
    import sys
    from neural_image_compression_v2_b200 import utils as U
    rng = np.random.default_rng(3)
    lut = rng.integers(0, 256, (5, 5, 5, 3)).astype(np.uint8)
    U.save_result_to_csv(lut, str(tmp_path / "a.csv"))
    text = (tmp_path / "a.csv").read_text()
    want = "".join("".join(f"{int(v)}," for v in lut[a, b].reshape(-1)) + "\n" for a in range(5) for b in range(5))
    assert text == want
    flt = torch.tensor(rng.random((3, 3, 3, 3)), dtype=torch.float32)
    U.save_result_to_csv(flt, str(tmp_path / "b.csv"))
    assert (tmp_path / "b.csv").read_text().split("\n")[0].split(",")[0] == str(flt[0, 0, 0, 0].item())
    d = tmp_path / "seq"
    assert U.make_filename_by_seq(str(d), "run_0.csv") == f"{d}/run_0_000.csv"
    (d / "run_0_000.csv").write_text("x")
    (d / "run_0_007.csv").write_text("x")
    assert U.make_filename_by_seq(str(d), "run_0.csv") == f"{d}/run_0_008.csv"
    from ref_loader import REF
    ref_utils = os.path.join(REF, "utils.py")
    if REF and os.path.exists(ref_utils):
        sys.dont_write_bytecode = True
        spec = importlib.util.spec_from_file_location("ref_utils_host", ref_utils)
        R = importlib.util.module_from_spec(spec)
        try:
            spec.loader.exec_module(R)
        except Exception:          # a missing optional import of the reference module: the format check above stands
            R = None
        if R is not None:
            R.save_result_to_csv(torch.tensor(lut), str(tmp_path / "ref.csv"))
            assert (tmp_path / "ref.csv").read_text() == text
            assert R.make_filename_by_seq(str(d), "run_0.csv") == U.make_filename_by_seq(str(d), "run_0.csv")
    cv2 = pytest.importorskip("cv2")
    movie = np.zeros((6, 32, 48, 3), dtype=np.uint8)
    for i in range(6):
        movie[i, :, : 8 * (i + 1)] = 200
    path = str(tmp_path / "m.avi")
    try:
        U.timelaps(movie, path, all_frame=6, width=48, height=32, frame_rate=8)
    except OSError:
        pytest.skip("this OpenCV build has no mp4v writer")
    back = U.readClip(path)
    assert back.shape == movie.shape and back.dtype == np.uint8
    assert np.abs(back.astype(np.int32) - movie.astype(np.int32)).mean() < 12.0        # lossy codec: same picture
    with pytest.raises(FileNotFoundError):
        U.readClip(str(tmp_path / "missing.avi"))
