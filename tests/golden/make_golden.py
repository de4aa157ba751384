"""Generate `tests/golden/*.npz|json` by executing the UNMODIFIED reference on seeded inputs.

Needs the reference project's `Projects/` directory:  NIC_REFERENCE_DIR=<it> python tests/golden/make_golden.py
The fixtures hold reference OUTPUTS; inputs are regenerated from seeds by `tests/golden/inputs.py`
(small inputs are stored as well, to make the fixtures self-describing).
Large outputs are stored as (flat index, value) subsamples + float64 column sums + a sha256 of the bytes.
"""
import contextlib
import hashlib
import io
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import inputs as I  # noqa: E402
from ref_loader import load_reference  # noqa: E402

torch.set_num_threads(8)
OUT = HERE


def quiet_load(*a, **k):
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        return load_reference(*a, **k)


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def T(a, grad=False):
    t = torch.tensor(np.asarray(a))
    return t.requires_grad_(True) if grad else t


def set_decoder(dec, params):
    sd = dec.state_dict()
    for key, p in zip(["decoder.0.weight", "decoder.0.bias", "decoder.2.weight", "decoder.2.bias",
                       "decoder.4.weight", "decoder.4.bias"], params):
        assert tuple(sd[key].shape) == p.shape, (key, sd[key].shape, p.shape)
        sd[key] = torch.tensor(p)
    dec.load_state_dict(sd)
    return dec


def sparse(a, count=4096):
    a = np.asarray(a)
    idx = I.subsample_index(a.shape, count)
    return idx.astype(np.int64), a.reshape(-1)[idx]


# --------------------------------------------------------------------------- tables / PE / quantisers
def gen_tables(g):
    fp_def = sys.modules["fp_def"]
    out = {}
    for s in (16, 32, 64, 128, 256, 512, 1024, 2048, 4096):
        out[str(s)] = {"levels": fp_def.return_pyramid_levels(s // 4),
                       "table": {str(k): v for k, v in dict(fp_def.create_pyramid_mip_levels(s, s // 4)).items()}}
    shapes = {}
    for s, dim in ((64, 2), (512, 2), (32, 3)):
        for no_mip in (True, False):
            fn = fp_def.create_pyramid if dim == 2 else fp_def.create_pyramid_3d
            pyr, lv = fn(s // 4, 12, 8, "cpu", torch.float32, no_mip)
            q_min = -(2 ** 8 - 1) / 2 ** 9
            assert all(float(p.min()) >= q_min and float(p.max()) <= 0.5 for p in pyr)
            shapes[f"{s}_{dim}_{int(no_mip)}"] = {"levels": lv, "shapes": [list(p.shape) for p in pyr]}
    out["pyramids"] = shapes
    with open(os.path.join(OUT, "tables.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)


def gen_pe():
    utils = sys.modules["utils"]
    rng = np.random.default_rng(7)
    c14 = np.array([[0, 1, 2, 3, 0, 0, 0, 0], [0, 0, 0, 0, 0, 1, 2, 3]], dtype=np.float32)   # test14.py input
    dy2 = (rng.integers(0, 8 * 600, (2, 512)) / 8.0).astype(np.float32)
    dy3 = (rng.integers(0, 8 * 80, (3, 512)) / 8.0).astype(np.float32)
    res = {"c14": c14, "dy2": dy2, "dy3": dy3}
    for name, c in (("c14", c14), ("dy2", dy2), ("dy3", dy3)):
        res[f"tri_{name}"] = utils.triangular_positional_encoding(T(c), 6, "cpu", torch.float32).numpy()
        res[f"sin_{name}"] = utils.positional_encoding(tuple(T(c)), 6, "cpu", torch.float32).numpy()
    res["tri4_dy2"] = utils.triangular_positional_encoding(T(dy2), 4, "cpu", torch.float32).numpy()
    np.savez(os.path.join(OUT, "pe.npz"), **res)


def gen_quant():
    models = sys.modules["models"]
    rng = np.random.default_rng(8)
    res = {}
    for bits in (8, 4, 2):
        q_min, q_max = I.q_range(bits)
        s = 2 ** bits - 1
        x = ((q_max - q_min) * rng.random(3000, dtype=np.float32) + np.float32(q_min)).astype(np.float32)
        ties = ((np.arange(-(2 ** (bits - 1)) + 1, 2 ** (bits - 1) + 1) - 0.5) / s).astype(np.float32)  # rounding ties
        edge = np.array([q_min, q_max, 0.0, -0.0, np.nextafter(np.float32(q_max), np.float32(0)),
                         np.nextafter(np.float32(q_min), np.float32(0))], dtype=np.float32)
        x = np.concatenate([x, ties, np.nextafter(ties, np.float32(1)), np.nextafter(ties, np.float32(-1)), edge])
        res[f"x{bits}"] = x
        res[f"q{bits}"] = models.quantize4fp(T(x), bits).numpy()
        res[f"code{bits}"] = models.save4fp(T(x), bits, torch.uint8).numpy()
        res[f"load{bits}"] = models.load4fp(T(res[f"code{bits}"]), bits, torch.float32).numpy()
        res[f"clamp{bits}"] = models.quantize_clamp(T(x * 1.5), bits).numpy()
    y = rng.random(4000, dtype=np.float32)
    y = np.concatenate([y, (np.arange(0, 256) + 0.5).astype(np.float32) / 255, np.array([0, 1], np.float32)])
    res["y"] = y
    res["y_to8"] = models.quantize_to_bit(T(y), 8).numpy()
    a = np.floor(rng.random((32, 32, 3)) * 256).astype(np.float32)
    b = np.clip(a + rng.integers(-3, 4, a.shape), 0, 255).astype(np.float32)
    utils = sys.modules["utils"]
    res["psnr_a"], res["psnr_b"] = a, b
    res["psnr"] = np.float64(utils.calculate_psnr(a, b))
    np.savez(os.path.join(OUT, "quant.npz"), **res)


# --------------------------------------------------------------------------- gather + decode (2-D)
def gen_2d():
    size, bits = 64, 8
    g = quiet_load(f"IMAGE_SIZE={size}", "TF_NO_MIP=0", "MAX_MIP_LEVEL=6")
    grids = I.make_grids(size, 2, bits=bits, seed=10)
    fp = [T(a) for a in grids]
    params = I.make_mlp(73, seed=11, gain=2.0)
    dec = set_decoder(g["ColorDecoder"](), params)
    res = {"image_size": size, "bits": bits}
    for i, a in enumerate(grids):
        res[f"grid{i}"] = a
    for i, p in enumerate(params):
        res[f"param{i}"] = p
    blocks = {0: (16, 40, 24), 1: (16, 8, 12), 2: (8, 3, 6), 3: (8, 0, 0), 4: (4, 0, 0), 5: (2, 0, 0), 6: (1, 0, 0)}
    with torch.no_grad():
        for mip in range(7):
            s, x, y = blocks[mip]
            res[f"X_block_mip{mip}"] = g["finally_decode_input_2d"](fp, s, mip, x, y).contiguous().numpy()
            res[f"block_mip{mip}"] = np.array([s, x, y])
            full = g["finally_decode_input_2d"](fp, size >> mip, mip).contiguous().numpy()
            res[f"X_full_sha_mip{mip}"] = sha(full)
            res[f"X_full_colsum_mip{mip}"] = full.astype(np.float64).sum(0)
            res[f"decode_mip{mip}"] = g["decode_image"](fp, dec, mip, False).numpy()
        # training-style builder, several crops, exercised through the sinusoidal switch too
        live = g["finally_decode_input_2d"].__globals__      # run_path hands back a COPY of the module globals
        live["TF_USE_TRI_PE"] = False
        res["X_block_sin_mip0"] = g["finally_decode_input_2d"](fp, 16, 0, 40, 24).contiguous().numpy()
        res["X_block_sin_mip3"] = g["finally_decode_input_2d"](fp, 8, 3, 0, 0).contiguous().numpy()
        live["TF_USE_TRI_PE"] = True
    np.savez(os.path.join(OUT, "gather_decode_2d.npz"), **res)

    # 4-bit and 2-bit quantised grids through decode (code parity feeds decode parity)
    res = {}
    for b in (4, 2):
        gq = I.make_grids(size, 2, bits=b, seed=20 + b, quantized=True)
        with torch.no_grad():
            res[f"decode_bits{b}"] = g["decode_image"]([T(a) for a in gq], dec, 0, False).numpy()
    np.savez(os.path.join(OUT, "decode_2d_lowbits.npz"), **res)


# --------------------------------------------------------------------------- gather + decode (3-D)
def gen_3d(method):
    size, bits = 32, 8
    vol = (I.make_image(size, 3, seed=30) * 255).astype(np.uint8).transpose(1, 2, 3, 0)   # [T,H,W,3]
    g = quiet_load(f"IMAGE_SIZE={size}", "IMAGE_DIMENSION=3", f"COMPRESSION_METHOD={method}", "TF_NO_MIP=1",
                   "CROP_MIP_LEVEL=3", npy=vol)   # the script's own 3-D mip branch breaks at its final PSNR (:487)
    cin = g["DECODER_INPUT_CHANNELS"]
    grids = I.make_grids(size, 3, bits=bits, seed=31)
    fp = [T(a) for a in grids]
    params = I.make_mlp(cin, seed=32, gain=2.0)
    dec = set_decoder(g["ColorDecoder"](), params)
    fin = g["finally_decode_input_3d" if method == 3 else "finally_decode_input_3d_v2"]
    cre = g["create_decoder_input_3d" if method == 3 else "create_decoder_input_3d_v2"]
    res = {"image_size": size, "bits": bits, "cin": cin}
    blocks = {0: (6, 7, 22, 13), 1: (6, 3, 9, 1), 2: (4, 1, 2, 3), 3: (4, 0, 0, 0), 4: (2, 0, 0, 0), 5: (1, 0, 0, 0)}
    with torch.no_grad():
        for mip in range(6):
            s, x, y, z = blocks[mip]
            res[f"X_block_mip{mip}"] = fin(fp, s, mip, x, y, z).contiguous().numpy()
            res[f"block_mip{mip}"] = np.array([s, x, y, z])
            if mip >= 1:
                res[f"decode_mip{mip}"] = g["decode_image"](fp, dec, mip, False).numpy()
            else:
                full = g["decode_image"](fp, dec, mip, False).numpy()
                res["decode_mip0_sha"] = sha(full)
                idx, val = sparse(full, 8192)
                res["decode_mip0_idx"], res["decode_mip0_val"] = idx, val
        coord = torch.tensor([[3, 11, 20], [24, 0, 7]])
        res["train_coord"] = coord.numpy()
        res["X_train_mip0"] = cre(fp, coord, 2, 0, 0).contiguous().numpy()     # 2 crops of 8^3
        res["X_train_mip1"] = cre(fp, coord // 2, 2, 0, 1).contiguous().numpy()  # 2 crops of 4^3
    np.savez(os.path.join(OUT, f"gather_decode_3d_m{method}.npz"), **res)
    return g


# --------------------------------------------------------------------------- training steps
def run_train(g, grids, params, mips, lods, coords, noises, t_max, bits, dim, method, num_crops):
    """Body of train_models (image_compression.py:220-269) with injected LOD / crop origins / noise."""
    fp = [T(a, grad=True) for a in grids]
    dec = set_decoder(g["ColorDecoder"](), params)
    opt = torch.optim.Adam([{"params": fp, "lr": 0.01}, {"params": dec.parameters(), "lr": 0.005}])
    sch = torch.optim.lr_scheduler.CosineAnnealingLR(opt, T_max=t_max, eta_min=0)
    crit = torch.nn.MSELoss()
    table = g["feature_pyramid_mip_levels_dict"]
    cre = {1: "create_decoder_input_2d", 3: "create_decoder_input_3d", 4: "create_decoder_input_3d_v2"}[method]
    fp_def = sys.modules["fp_def"]
    losses, first_grads, frozen = [], None, False
    for epoch, lod in enumerate(lods):
        if epoch > t_max * 0.95 and not frozen:          # image_compression.py:227-231
            fp_def.fp_freeze(fp)
            fp = fp_def.fp_all_quantize(fp, bits)
            frozen = True
        fl = table[lod]
        coord = torch.tensor(coords[epoch])
        data = T(mips[lod])
        crop = 2 ** max(0, (8 if method == 1 else g["CROP_MIP_LEVEL"]) - lod)
        tg = []
        for c in coords[epoch]:                          # image_compression.py:39-48
            sl = (slice(None),) + tuple(slice(int(c[a]), int(c[a]) + crop) for a in range(dim))
            tg.append(data[sl].reshape(3, -1).T)
        target = torch.stack(tg).reshape(-1, 3)
        x = g[cre](fp, coord, num_crops, fl, lod)
        if epoch < t_max * 0.95:
            x = x + T(noises[epoch])
        out = dec(x)
        loss = crit(out, target)
        opt.zero_grad()
        loss.backward()
        if first_grads is None:
            first_grads = {"g0": fp[2 * fl].grad.numpy().copy(), "g1": fp[2 * fl + 1].grad.numpy().copy(),
                           "mlp": [p.grad.numpy().copy() for p in dec.parameters()], "out": out.detach().numpy().copy()}
        opt.step()
        sch.step()
        fp_def.fp_quantize_clamp(fp, fl, bits)
        losses.append(float(loss.item()))
    return losses, first_grads, [a.detach().numpy() for a in fp], [p.detach().numpy() for p in dec.parameters()]


def gen_train_2d():
    size, bits, nc = 512, 8, 2
    g = quiet_load(f"IMAGE_SIZE={size}", "TF_NO_MIP=0", "MAX_MIP_LEVEL=9")
    grids = I.make_grids(size, 2, bits=bits, seed=40)
    params = I.make_mlp(73, seed=41)
    mips = I.box_mips(I.make_image(size, 2, seed=42), 9)
    rng = np.random.default_rng(43)
    t_max = 40
    lods = [3, 4, 3, 5, 2, 6, 3, 4] * 5               # 40 steps: last one trains on frozen, quantised grids
    coords, noises = [], []
    for e, lod in enumerate(lods):
        crop = 2 ** (8 - lod)
        coords.append(rng.integers(0, (size >> lod) - crop + 1, (nc, 2)))
        noises.append(I.make_noise(nc * crop * crop, 73, bits, 1000 + e))
    losses, fg, fp, pr = run_train(g, grids, params, mips, lods, coords, noises, t_max, bits, 2, 1, nc)
    res = {"lods": np.array(lods), "losses": np.array(losses), "nc": nc, "t_max": t_max, "size": size}
    for e, c in enumerate(coords):
        res[f"coord{e}"] = c
    for i, p in enumerate(pr):
        res[f"param{i}"] = p
    for i, p in enumerate(fg["mlp"]):
        res[f"grad0_param{i}"] = p
    res["grad0_g0_idx"], res["grad0_g0_val"] = sparse(fg["g0"], 8192)
    res["grad0_g1_idx"], res["grad0_g1_val"] = sparse(fg["g1"], 8192)
    res["grad0_g0_sum"], res["grad0_g1_sum"] = fg["g0"].astype(np.float64).sum(), fg["g1"].astype(np.float64).sum()
    res["grad0_g0_abs"], res["grad0_g1_abs"] = np.abs(fg["g0"]).astype(np.float64).sum(), np.abs(fg["g1"]).astype(np.float64).sum()
    res["out0_idx"], res["out0_val"] = sparse(fg["out"], 4096)
    for i, a in enumerate(fp):
        res[f"grid{i}_idx"], res[f"grid{i}_val"] = sparse(a, 8192)
        res[f"grid{i}_sum"] = a.astype(np.float64).sum()
    np.savez(os.path.join(OUT, "train_2d.npz"), **res)

    # default config shape (TF_NO_MIP=True semantics: lod 0, 256^2 crops, step 1/4), two steps
    lods = [0, 0]
    coords = [rng.integers(0, size - 256 + 1, (nc, 2)) for _ in lods]
    noises = [I.make_noise(nc * 256 * 256, 73, bits, 2000 + e) for e in range(2)]
    losses, fg, fp, pr = run_train(g, grids, params, mips, lods, coords, noises, 1000, bits, 2, 1, nc)
    res = {"lods": np.array(lods), "losses": np.array(losses), "nc": nc, "t_max": 1000, "size": size}
    for e, c in enumerate(coords):
        res[f"coord{e}"] = c
    for i, p in enumerate(pr):
        res[f"param{i}"] = p
    for i, p in enumerate(fg["mlp"]):
        res[f"grad0_param{i}"] = p
    res["grad0_g0_idx"], res["grad0_g0_val"] = sparse(fg["g0"], 8192)
    res["grad0_g1_idx"], res["grad0_g1_val"] = sparse(fg["g1"], 8192)
    for i in (0, 1):
        res[f"grid{i}_idx"], res[f"grid{i}_val"] = sparse(fp[i], 8192)
        res[f"grid{i}_sum"] = fp[i].astype(np.float64).sum()
    np.savez(os.path.join(OUT, "train_2d_lod0.npz"), **res)


def gen_train_3d(method):
    size, bits, nc = 32, 8, 2
    vol = (I.make_image(size, 3, seed=30) * 255).astype(np.uint8).transpose(1, 2, 3, 0)
    g = quiet_load(f"IMAGE_SIZE={size}", "IMAGE_DIMENSION=3", f"COMPRESSION_METHOD={method}", "TF_NO_MIP=1",
                   "CROP_MIP_LEVEL=3", npy=vol)   # the script's own 3-D mip branch breaks at its final PSNR (:487)
    cin = g["DECODER_INPUT_CHANNELS"]
    grids = I.make_grids(size, 3, bits=bits, seed=50)
    params = I.make_mlp(cin, seed=51)
    data = [g["images"][0].numpy()] * 6                 # the reference's own [3,T,H,W]/256 target; its 3-D "mips"
    #                                                     are all the same full-size volume (image_compression.py:470-477)
    rng = np.random.default_rng(53)
    t_max = 12
    lods = [0, 1, 0, 2, 0, 1, 0, 0, 1, 0, 2, 0]
    coords, noises = [], []
    for e, lod in enumerate(lods):
        crop = 2 ** (3 - lod)
        coords.append(rng.integers(0, (size >> lod) - crop + 1, (nc, 3)))
        noises.append(I.make_noise(nc * crop ** 3, cin, bits, 3000 + e))
    losses, fg, fp, pr = run_train(g, grids, params, data, lods, coords, noises, t_max, bits, 3, method, nc)
    res = {"lods": np.array(lods), "losses": np.array(losses), "nc": nc, "t_max": t_max, "size": size, "cin": cin,
           "target": data[0]}
    for e, c in enumerate(coords):
        res[f"coord{e}"] = c
    for i, p in enumerate(pr):
        res[f"param{i}"] = p
    for i, p in enumerate(fg["mlp"]):
        res[f"grad0_param{i}"] = p
    res["grad0_g0"], res["grad0_g1"] = fg["g0"], fg["g1"]
    for i, a in enumerate(fp):
        res[f"grid{i}"] = a
    np.savez_compressed(os.path.join(OUT, f"train_3d_m{method}.npz"), **res)


if __name__ == "__main__":
    g = quiet_load("IMAGE_SIZE=64")
    gen_tables(g)
    gen_pe()
    gen_quant()
    gen_2d()
    gen_3d(3)
    gen_3d(4)
    gen_train_2d()
    gen_train_3d(3)
    gen_train_3d(4)
    for f in sorted(os.listdir(OUT)):
        if f.endswith((".npz", ".json")):
            print(f, os.path.getsize(os.path.join(OUT, f)))
