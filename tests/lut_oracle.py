"""numpy oracle of applying a baked colour LUT (nic_lut_apply, include/nic.h), float32 step by step in the GPU's order so that
it reproduces the fp32 arm bit for bit: the trilinear arm takes its taps and weights from sample_oracle.tap_rule, the
tetrahedral arm restates tetra_corners (nic_common.cuh)."""
import numpy as np

from sample_oracle import tap_rule

F32 = np.float32


def unit_coords(image):
    """Pixels [..., 3] -> normalised coordinates [P, 3] float32: uint8 v as v / 255 (one correctly rounded division, as
    __fdiv_rn), float32 as given."""
    c = np.asarray(image).reshape(-1, 3)
    if c.dtype == np.uint8:
        return (c.astype(F32) / F32(255)).astype(F32)
    return c.astype(F32)


def axis_rule(u, extent):
    """Per axis: (fraction f float32 [P, 3], low taps, high taps int64 [P, 3]) of the align_corners / clamp rule."""
    f = np.zeros(u.shape, F32)
    lo = np.zeros(u.shape, np.int64)
    hi = np.zeros(u.shape, np.int64)
    for a in range(3):
        s = int(extent[a])
        p = (u[:, a] * F32(s - 1)).astype(F32)
        p = np.fmin(np.fmax(p, F32(-2.0 ** 24)), F32(2.0 ** 24))          # NaN -> -2^24 (fmax ignores a NaN operand)
        i0 = np.floor(p)
        f[:, a] = (p - i0).astype(F32)
        lo[:, a] = np.clip(i0.astype(np.int64), 0, s - 1)
        hi[:, a] = np.clip(i0.astype(np.int64) + 1, 0, s - 1)
    return f, lo, hi


def trilinear(dense, u):
    """dense [Sx, Sy, Sz, C] float32, u [P, 3] float32 -> [P, C] float32: acc = 0, acc = acc + w_k * v_k over the 8 taps."""
    dense = np.asarray(dense, F32)
    taps, w = tap_rule(u, dense.shape[:3], True, "clamp")
    acc = np.zeros((u.shape[0], dense.shape[3]), F32)
    for k in range(8):
        v = dense[taps[:, k, 0], taps[:, k, 1], taps[:, k, 2]]
        acc = (acc + (w[:, k, None] * v).astype(F32)).astype(F32)
    return acc


def tetra_corners(u, extent):
    """(corners int64 [P, 4, 3], weights float32 [P, 4]) of the tetrahedral rule: axes by descending fraction (stable, so
    ties keep x before y before z), corners lo, + e_a1, + e_a2, hi; weights 1 - f_a1, f_a1 - f_a2, f_a2 - f_a3, f_a3."""
    f, lo, hi = axis_rule(u, extent)
    order = np.argsort(-f, axis=1, kind="stable")
    fs = np.take_along_axis(f, order, 1)
    w = np.stack([(F32(1) - fs[:, 0]).astype(F32), (fs[:, 0] - fs[:, 1]).astype(F32), (fs[:, 1] - fs[:, 2]).astype(F32),
                  fs[:, 2]], 1)
    corners = np.repeat(lo[:, None, :], 4, 1)
    rows = np.arange(u.shape[0])
    for k in range(1, 4):
        for j in range(k, 4):
            corners[rows, j, order[:, k - 1]] = hi[rows, order[:, k - 1]]
    return corners, w


def tetrahedral(dense, u):
    """dense [Sx, Sy, Sz, C] float32, u [P, 3] float32 -> [P, C] float32: acc = 0, acc = acc + w_k * v_k, k = 0..3."""
    dense = np.asarray(dense, F32)
    corners, w = tetra_corners(u, dense.shape[:3])
    acc = np.zeros((u.shape[0], dense.shape[3]), F32)
    for k in range(4):
        v = dense[corners[:, k, 0], corners[:, k, 1], corners[:, k, 2]]
        acc = (acc + (w[:, k, None] * v).astype(F32)).astype(F32)
    return acc


def apply(dense, image, interpolation):
    u = unit_coords(image)
    return trilinear(dense, u) if interpolation == "trilinear" else tetrahedral(dense, u)


def to_u8(v):
    """floor(v * 255 + .5) with a separate float32 multiply and add, clamped to [0, 255]."""
    q = np.floor(((np.asarray(v, F32) * F32(255)).astype(F32) + F32(0.5)).astype(F32))
    return np.clip(q, 0, 255).astype(np.uint8)
