"""Full-scale and 12-bit inputs for motion compensation, chroma-from-luma, CDEF and the RDO
distortions: the shared input builders, and the CPU checks that pin the oracle to plain int64 /
Python-integer models at the ranges where the arithmetic runs out of bits.

The parity tests elsewhere feed these kernels uniform noise or small differences, so the i16 MC
intermediate, the i16 CfL samples, CDEF's high-bit-depth direction search and the wrapping casts of
the distortions never see their limits there.  The builders here produce what real content can
reach: pixels that follow the sign of the MC filter taps, full-scale luma, unshifted 10/12-bit
noise, 0/max planes and block pairs at full contrast.  tests/test_zz_full_scale_pred_gpu.py runs the
same inputs through the CUDA kernels."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from tests import oracle_lib as O
from tests.test_full_scale import pixel_dtype
from tests.test_oracle_cdef_spec import spec_direction, spec_filter
from tests.test_oracle_rdo_dist import L as RL

BDS = [8, 10, 12]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def rnd(v, b):
    """(v + 2^(b-1)) >> b on Python ints / int64 arrays (arithmetic shift)"""
    return (v + ((1 << b) >> 1)) >> b


def ib_of(bd):
    """intermediate bits of the MC passes (mc.rs:258): 4, and 2 at 12 bit"""
    return 2 if bd == 12 else 4


def prep_bias(bd):
    return 0 if bd == 8 else 8192


# ---------------------------------------------------------------- MC: the filter table and its bounds

def filter_table():
    """kSubpel[6][16][8] as written in rav1e_b200/csrc/mc_filters.cuh (768 values)"""
    text = open(os.path.join(ROOT, "rav1e_b200", "csrc", "mc_filters.cuh")).read()
    body = text[text.index("kSubpel[6][16][8]"):]
    body = body[body.index("{"):body.index("};")]
    vals = [int(v) for v in re.findall(r"-?\d+", body)]
    assert len(vals) == 768
    return np.array(vals, np.int64).reshape(6, 16, 8)


def filter_bank(mode, length):
    """mc.rs:238-247: 4-tap banks 4/5 for REGULAR/SMOOTH(/SHARP -> REGULAR) when the length is <= 4"""
    return mode if (mode == 3 or length > 4) else min(mode, 1) + 4


def taps(mode, frac, length):
    return filter_table()[filter_bank(mode, length)][frac]


def h_bounds(row, bd):
    """(min, max) of the H pass round(sum, 7 - ib) of filter row `row` over pixels in [0, max]"""
    m = (1 << bd) - 1
    pos, neg = int(row[row > 0].sum()), int(row[row < 0].sum())
    r0 = 7 - ib_of(bd)
    return rnd(m * neg, r0), rnd(m * pos, r0)


def hv_bounds(fx, fy, bd):
    """(min, max) of the V-pass sum over an intermediate at the H-pass extremes of fx"""
    lo, hi = h_bounds(fx, bd)
    vmax = sum(int(t) * (hi if t > 0 else lo) for t in fy)
    vmin = sum(int(t) * (lo if t > 0 else hi) for t in fy)
    return vmin, vmax


def table_bounds(bd):
    """over all 96 rows of the table: the H-pass intermediate's (min, max), and the pre-bias HV prep
    value round(V, 7)'s (min, max)"""
    tab = filter_table().reshape(-1, 8)
    hs = [h_bounds(r, bd) for r in tab]
    hv = [hv_bounds(fx, fy, bd) for fx in tab for fy in tab]
    return (min(h[0] for h in hs), max(h[1] for h in hs),
            rnd(min(v[0] for v in hv), 7), rnd(max(v[1] for v in hv), 7))


# measured from the table by test_mc_table_bounds_fit_i16 below
H_BOUNDS = {8: (-1785, 5865), 10: (-7161, 23529), 12: (-7166, 23546)}
PREP_PREBIAS = {8: (-5132, 9212), 10: (-20588, 36956), 12: (-20602, 36983)}


def tap_sign_tile(fx, fy, w, h, bd, sign):
    """(h+7) x (w+7) tile, period 8: max where sign(fy[r]) * sign(fx[c]) == sign, else 0 (zero taps
    take 0).  At every output (8i, 8j) the H pass of a row with fy > 0 reaches its extreme of the
    sign, and the V pass its extreme of the sign: sign +1 drives the HV sum to its maximum, -1 to its
    minimum."""
    m = (1 << bd) - 1
    s = np.outer(np.sign(fy), np.sign(fx)) * sign
    base = np.where(s > 0, m, 0)
    return np.ascontiguousarray(np.tile(base, ((h + 14) // 8, (w + 14) // 8))[:h + 7, :w + 7].astype(pixel_dtype(bd)))


def h_only_tile(fx, w, h, bd, sign):
    """one row pattern repeated: every row's H pass at its extreme of `sign`"""
    m = (1 << bd) - 1
    row = np.where(np.sign(fx) * sign > 0, m, 0)
    row = np.tile(row, (w + 14) // 8)[:w + 7]
    return np.ascontiguousarray(np.tile(row, (h + 7, 1)).astype(pixel_dtype(bd)))


def const_tile(w, h, bd, v):
    return np.full((h + 7, w + 7), v, pixel_dtype(bd))


def checker_tile(w, h, bd, phase=0):
    m = (1 << bd) - 1
    return np.ascontiguousarray(((np.indices((h + 7, w + 7)).sum(0) + phase) & 1).astype(pixel_dtype(bd)) * m)


def mc_tiles(fx, fy, w, h, bd):
    """every MC input for one filter pair: the tap-sign tiles of both signs, the H-only patterns of
    both signs, constant 0 and max, and a 0/max checkerboard in both phases"""
    m = (1 << bd) - 1
    return [tap_sign_tile(fx, fy, w, h, bd, 1), tap_sign_tile(fx, fy, w, h, bd, -1),
            h_only_tile(fx, w, h, bd, 1), h_only_tile(fx, w, h, bd, -1), const_tile(w, h, bd, 0),
            const_tile(w, h, bd, m), checker_tile(w, h, bd), checker_tile(w, h, bd, 1)]


def mc_model(tile, fx, fy, w, h, bd):
    """int64 two-pass model of put_8tap / prep_8tap on the block whose footprint is `tile`: H pass
    rounded by 7 - ib into an intermediate of h + 7 rows (the identity row at fraction 0 leaves
    px << ib), V pass; put rounds by 7 + ib and clips, prep rounds by 7 and subtracts the bias.
    Returns (put, prep before the bias, intermediate)."""
    ib = ib_of(bd)
    t = tile.astype(np.int64)
    inter = rnd(sum(int(fx[k]) * t[:h + 7, k:k + w] for k in range(8)), 7 - ib)
    v = sum(int(fy[k]) * inter[k:k + h] for k in range(8))
    put = np.clip(rnd(v, 7 + ib), 0, (1 << bd) - 1)
    return put, rnd(v, 7), inter


def mc_avg_model(t1, t2, bd):
    ib = ib_of(bd)
    return np.clip(rnd(t1.astype(np.int64) + t2 + 2 * prep_bias(bd), ib + 1), 0, (1 << bd) - 1)


def mc_fracs(step=1):
    """(col_frac, row_frac): copy, every H-only and V-only fraction, and the HV pairs (f, f) and
    (f, 16 - f); with step 2 only the even fractions (what a luma vector can address)"""
    fs = range(step, 16, step)
    return ([(0, 0)] + [(f, 0) for f in fs] + [(0, f) for f in fs] + [(f, f) for f in fs]
            + [(f, 16 - f) for f in fs if f != 8])


MODE_PAIRS = [(mx, my) for mx in range(4) for my in range(4)]


def oracle_put_prep(tile, w, h, cf, rf, mx, my, bd):
    p = O.Plane(w + 7, h + 7, 0, tile.dtype)
    p.fill_from(tile)
    return (O.put_8tap(p, 3, 3, w, h, cf, rf, mx, my, bd), O.prep_8tap(p, 3, 3, w, h, cf, rf, mx, my, bd))


def test_mc_filter_table_is_the_oracles():
    """The 768 values of mc_filters.cuh are the rows the oracle filters with, for every mode,
    fraction and block length (4-tap banks at <= 4)."""
    L = O.lib()
    f = (C.c_int32 * 8)()
    for mode in range(4):
        for length in (2, 4, 8, 16):
            for frac in range(16):
                L.orc_get_filter(mode, frac, length, f)
                assert list(f) == taps(mode, frac, length).tolist(), (mode, frac, length)


@pytest.mark.parametrize("bd", BDS)
def test_mc_table_bounds_fit_i16(bd):
    """The H-pass intermediate extremes over the table, and the pre-bias HV prep value: the
    intermediate fits i16 with room to spare (so its `as i16` never truncates); the prep value
    exceeds i16 before the 8192 bias at 10/12 bit and fits after it."""
    hmin, hmax, pmin, pmax = table_bounds(bd)
    print(f"\n{bd}-bit: H-pass intermediate in [{hmin}, {hmax}], HV prep before the bias in [{pmin}, {pmax}]")
    assert (hmin, hmax) == H_BOUNDS[bd]
    assert (pmin, pmax) == PREP_PREBIAS[bd]
    assert -(1 << 15) <= hmin and hmax < 1 << 15
    assert -(1 << 15) <= pmin - prep_bias(bd) and pmax - prep_bias(bd) < 1 << 15
    if bd > 8:
        assert pmax >= 1 << 15                       # the order of bias and cast matters


@pytest.mark.parametrize("bd", BDS)
def test_mc_oracle_against_int64_model(bd):
    """Oracle put_8tap / prep_8tap == mc_model on every tile of mc_tiles, all 16 mode pairs, copy /
    H-only / V-only / HV fractions, 8x8 (8-tap banks) and 4x4 (4-tap banks); mc_avg == its model on
    the extreme preps in both sign combinations.  The tap-sign tiles reach the table's bounds."""
    seen_h, seen_p = [0, 0], [0, 0]
    for w, h in ((8, 8), (4, 4)):
        for mx, my in MODE_PAIRS:
            for cf, rf in mc_fracs():
                fx, fy = taps(mx, cf, w), taps(my, rf, h)
                preps = []
                for k, tile in enumerate(mc_tiles(fx, fy, w, h, bd)):
                    put, pre, inter = mc_model(tile, fx, fy, w, h, bd)
                    prep = pre - prep_bias(bd)
                    assert prep.min() >= -(1 << 15) and prep.max() < 1 << 15
                    got_put, got_prep = oracle_put_prep(tile, w, h, cf, rf, mx, my, bd)
                    ctx = (w, h, mx, my, cf, rf, k)
                    np.testing.assert_array_equal(got_put, put, err_msg=str(ctx))
                    np.testing.assert_array_equal(got_prep, prep, err_msg=str(ctx))
                    seen_h = [min(seen_h[0], int(inter.min())), max(seen_h[1], int(inter.max()))]
                    seen_p = [min(seen_p[0], int(pre.min())), max(seen_p[1], int(pre.max()))]
                    if k < 2 and cf and rf:
                        vmin, vmax = hv_bounds(fx, fy, bd)
                        want = rnd(vmax, 7) if k == 0 else rnd(vmin, 7)
                        assert pre[0, 0] == want, ctx       # the tile drives output (0, 0) to the bound
                    preps.append(got_prep)
                for a, b in ((0, 0), (0, 1), (1, 1), (1, 0)):
                    np.testing.assert_array_equal(O.mc_avg(preps[a], preps[b], bd),
                                                  mc_avg_model(preps[a], preps[b], bd))
    assert tuple(seen_h) == H_BOUNDS[bd]
    assert tuple(seen_p) == PREP_PREBIAS[bd]


# ---------------------------------------------------------------- CfL at full scale

LAYOUTS = [(1, 1), (1, 0), (0, 0)]
CFL_SIZES = [(4, 4), (8, 8), (16, 16), (32, 32), (8, 4), (4, 8), (16, 8), (8, 16), (32, 16), (16, 32),
             (4, 16), (16, 4), (8, 32), (32, 8)]


def cfl_lumas(lw, lh, bd, xdec, ydec):
    """full-scale luma blocks (lh x lw): constant max, a 0/max checkerboard, vertical and horizontal
    steps, one max subsampling footprint in a 0 block and one 0 footprint in a max block"""
    m = (1 << bd) - 1
    dt = pixel_dtype(bd)
    out = [np.full((lh, lw), m), (np.indices((lh, lw)).sum(0) & 1) * m]
    v = np.zeros((lh, lw), np.int64)
    v[:, lw // 2:] = m
    hs = np.zeros((lh, lw), np.int64)
    hs[lh // 2:] = m
    out += [v, hs]
    spot = np.zeros((lh, lw), np.int64)
    spot[:1 << ydec, :1 << xdec] = m
    out += [spot, m - spot]
    return [np.ascontiguousarray(x.astype(dt)) for x in out]


def cfl_ac_model(luma, bw, bh, w_pad, h_pad, xdec, ydec):
    """predict.rs:1020-1063 on int64: the subsampled sum << (3 - xdec - ydec) of the clamped
    position, minus the rounded average.  Returns (ac, samples before the average)."""
    L = luma.astype(np.int64)
    max_w, max_h = (bw - w_pad * 4) << xdec, (bh - h_pad * 4) << ydec
    mx, my = max(max_w, 8) - (1 << xdec), max(max_h, 8) - (1 << ydec)
    ys = np.minimum(np.arange(bh) << ydec, my)
    xs = np.minimum(np.arange(bw) << xdec, mx)
    s = L[ys][:, xs]
    if xdec:
        s = s + L[ys][:, xs + 1]
    if ydec:
        s = s + L[ys + 1][:, xs] + L[ys + 1][:, xs + 1]
    s = s << (3 - xdec - ydec)
    shift = (bw.bit_length() - 1) + (bh.bit_length() - 1)
    avg = rnd(int(s.sum()), shift)
    return (s - avg).reshape(-1), s


def cfl_pads(bw, bh, xdec, ydec):
    """the w_pad / h_pad in 0..3 that leave at least one 4-wide column / row of real luma"""
    return [(wp, hp) for wp in range(4) for hp in range(4) if 4 * wp < bw and 4 * hp < bh]


def test_cfl_ac_oracle_at_12_bit():
    """Oracle pred_cfl_ac == cfl_ac_model at 12 bit for every layout, block size 4x4 .. 32x32 and
    valid padding; the subsampled sample reaches 8 * 4095 = 32760 (7 below the i16 limit) and ac its
    largest magnitudes, one footprint against a flat block."""
    lo = hi = top = 0
    for xdec, ydec in LAYOUTS:
        for bw, bh in CFL_SIZES:
            for w_pad, h_pad in cfl_pads(bw, bh, xdec, ydec):
                for luma in cfl_lumas(bw << xdec, bh << ydec, 12, xdec, ydec):
                    want, s = cfl_ac_model(luma, bw, bh, w_pad, h_pad, xdec, ydec)
                    got = O.pred_cfl_ac(luma, bw, bh, w_pad, h_pad, xdec, ydec)
                    np.testing.assert_array_equal(got, want, err_msg=f"{bw}x{bh} dec {xdec}{ydec} pad {w_pad}{h_pad}")
                    top = max(top, int(s.max()))
                    lo, hi = min(lo, int(want.min())), max(hi, int(want.max()))
    print(f"\n12-bit CfL: samples up to {top}, ac in [{lo}, {hi}]")
    assert top == 8 * 4095 == 32760
    # one footprint at max in a 0 block of 32x32 samples: 32760 - round(32760 / 1024); and the reverse
    assert (lo, hi) == (-32728, 32728)


def scaled_luma_q0(alpha, ac):
    """predict.rs:626-635: round(|alpha * ac| / 64) with the sign of the product"""
    p = alpha * ac.astype(np.int64)
    return np.sign(p) * ((np.abs(p) + 32) >> 6)


def dc_model(edge, variant, w, h, bd):
    """DC_128 / DC_LEFT / DC_TOP / DC (predict.rs:786-840) on the IntraEdge buffer (top-left at 128)"""
    above = edge[129:129 + w].astype(np.int64)
    left = edge[128 - h:128].astype(np.int64)
    if variant == 0:
        return 128 << (bd - 8)
    if variant == 1:
        return (int(left.sum()) + (h >> 1)) // h
    if variant == 2:
        return (int(above.sum()) + (w >> 1)) // w
    return (int(above.sum() + left.sum()) + ((w + h) >> 1)) // (w + h)


def cfl_pred_model(edge, variant, ac, alpha, w, h, bd):
    """predict.rs:1065-1088: DC plus the scaled ac, clipped to [0, max]; alpha 0 leaves the DC"""
    dc = dc_model(edge, variant, w, h, bd)
    if alpha == 0:
        return np.full((h, w), dc)
    return np.clip(dc + scaled_luma_q0(alpha, ac).reshape(h, w), 0, (1 << bd) - 1)


def cfl_edges(bd):
    """IntraEdge buffers: all 0, all max, above max / left 0, and alternating 0/max"""
    m = (1 << bd) - 1
    dt = pixel_dtype(bd)
    e = [np.zeros(O.EDGE_LEN), np.full(O.EDGE_LEN, m), np.where(np.arange(O.EDGE_LEN) > 128, m, 0),
         (np.arange(O.EDGE_LEN) & 1) * m]
    return [np.ascontiguousarray(x.astype(dt)) for x in e]


def cfl_ac_inputs(bd):
    """(bw, bh, ac) of extreme ac blocks: the 4:4:4 lumas of cfl_lumas at 8x8, 16x8 and 32x32"""
    out = []
    for bw, bh in ((8, 8), (16, 8), (32, 32)):
        for luma in cfl_lumas(bw, bh, bd, 0, 0):
            out.append((bw, bh, O.pred_cfl_ac(luma, bw, bh, 0, 0, 0, 0)))
    return out


def test_cfl_prediction_oracle_at_12_bit():
    """Oracle UV_CFL_PRED == cfl_pred_model at 12 bit: every alpha in -16..16, all four DC variants,
    edges at 0, at max and mixed, on extreme ac blocks.  The unclipped value leaves [0, 4095] on both
    sides, so the clip at the 12-bit maximum is what the output shows."""
    bd = 12
    M = O.MODES.index("UV_CFL_PRED")
    clipped_hi = clipped_lo = 0
    for bw, bh, ac in cfl_ac_inputs(bd):
        for ei, edge in enumerate(cfl_edges(bd)):
            for variant in range(4):
                for alpha in range(-16, 17):
                    want = cfl_pred_model(edge, variant, ac, alpha, bw, bh, bd)
                    got = O.predict_intra(M, variant, edge, bw, bh, bd, angle=alpha, ac=ac, left_len=bh, above_len=bw)
                    np.testing.assert_array_equal(got, want, err_msg=f"{bw}x{bh} edge {ei} var {variant} alpha {alpha}")
                    raw = dc_model(edge, variant, bw, bh, bd) + scaled_luma_q0(alpha, ac)
                    clipped_hi += int((raw > 4095).sum())
                    clipped_lo += int((raw < 0).sum())
                    assert (got[raw.reshape(bh, bw) > 1023] > 1023).all()
    assert clipped_hi and clipped_lo


# ---------------------------------------------------------------- CDEF at high bit depth

def cdef_planes(W, H, bd, seed):
    """named full-scale CDEF inputs: uniform full-range noise (low bits set), 0/max checkerboard,
    vertical and horizontal 0/max stripes (the largest `var`), and step edges at the frame border
    (max pixels next to the sentinel outside the frame)"""
    m = (1 << bd) - 1
    rng = np.random.default_rng(seed)
    yy, xx = np.indices((H, W))
    out = {"noise": rng.integers(0, m + 1, (H, W)),
           "checker": ((yy + xx) & 1) * m,
           "vstripes": ((xx >> 1) & 1) * m,
           "hstripes": (yy & 1) * m,
           "border": np.where((xx < 3) | (yy < 3) | (xx >= W - 3) | (yy >= H - 3), m, 0)}
    return {k: np.ascontiguousarray(v.astype(pixel_dtype(bd))) for k, v in out.items()}


@pytest.mark.parametrize("bd", [10, 12])
def test_cdef_direction_sees_only_the_top_8_bits(bd):
    """Oracle cdef_find_dir of an HBD block == cdef_find_dir of block >> (bd - 8) at 8 bit (direction
    and variance), and == the specification's direction process, on unshifted noise, full-contrast
    patterns and noise with the low bits only."""
    rng = np.random.default_rng(bd)
    m = (1 << bd) - 1
    blocks = []
    for name, p in cdef_planes(64, 64, bd, bd).items():
        blocks += [p[y:y + 8, x:x + 8] for y in (0, 8, 24) for x in (0, 16, 40)]
    blocks += [rng.integers(0, 1 << (bd - 8), (8, 8)) + (rng.integers(0, 256, (8, 8)) << (bd - 8)) for _ in range(40)]
    blocks += [rng.integers(0, m + 1, (8, 8)) for _ in range(200)]
    for blk in blocks:
        blk = np.ascontiguousarray(np.asarray(blk).astype(np.uint16))
        want = O.cdef_find_dir(np.ascontiguousarray((blk >> (bd - 8)).astype(np.uint8)), 8)
        assert O.cdef_find_dir(blk, bd) == want
        assert spec_direction(blk, bd) == want


def cdef_filter_blocks(bd, seed):
    """12 x 12 tiles (block at [2:10, 2:10]): unshifted noise, 0/max checkerboard and stripes, one
    max pixel in 0 and one 0 pixel in max"""
    m = (1 << bd) - 1
    rng = np.random.default_rng(seed)
    yy, xx = np.indices((12, 12))
    spot = np.zeros((12, 12), np.int64)
    spot[5, 6] = m
    out = [rng.integers(0, m + 1, (12, 12)), ((yy + xx) & 1) * m, (xx & 1) * m, ((yy >> 1) & 1) * m, spot, m - spot]
    return [np.ascontiguousarray(x.astype(pixel_dtype(bd))) for x in out]


@pytest.mark.parametrize("bd", [10, 12])
@pytest.mark.parametrize("xdec,ydec", [(0, 0), (1, 1), (1, 0)])
def test_cdef_filter_oracle_at_full_scale(bd, xdec, ydec):
    """Oracle cdef_filter_block == the specification's filter process on unshifted HBD data and
    full-contrast blocks at pri 15 / sec 4 (scaled by the bit depth), damping 3 and 6, all 16 edge
    masks (each with its own direction)."""
    L = O.lib()
    cs = bd - 8
    w, h = 8 >> xdec, 8 >> ydec
    for k, img in enumerate(cdef_filter_blocks(bd, 40 + bd)):
        for base_damping in (3, 6):
            damping = base_damping + cs - (1 if xdec else 0)
            for pri, sec in ((15 << cs, 4 << cs), (15 << cs, 0), (0, 4 << cs)):
                for edges in range(16):
                    d = (edges + k + base_damping) & 7
                    dst = np.zeros((h, w), img.dtype)
                    L.orc_cdef_filter_block_px(O.ptr(dst), w, O.ptr(img, 2 * 12 + 2), 12, img.itemsize, pri, sec, d,
                                               damping, bd, xdec, ydec, edges)
                    want = spec_filter(img, w, h, pri, sec, d, damping, bd, edges)
                    np.testing.assert_array_equal(dst, want, err_msg=f"block {k} damping {damping} pri {pri} "
                                                  f"sec {sec} edges {edges} d {d}")


# ---------------------------------------------------------------- RDO distortions in Python integers

U32, U64 = 1 << 32, 1 << 64
SCALES = [1, 1 << 14, (1 << 28) - 1]       # DistortionScale: the smallest, unity, the largest (rdo.rs:574-576)
WSSE_SIZES = [(w, h) for w in (4, 8, 16, 32, 64, 128) for h in (4, 8, 16, 32, 64, 128) if max(w, h) <= 4 * min(w, h)]


def block_pairs(w, h, bd):
    """(name, a, b) at full contrast: 0 vs max, max vs 0, a checkerboard vs its inverse, a checkerboard
    vs a flat 0 and vs a flat max block, and a single max pixel against 0"""
    m = (1 << bd) - 1
    dt = pixel_dtype(bd)
    z, f = np.zeros((h, w), np.int64), np.full((h, w), m)
    chk = (np.indices((h, w)).sum(0) & 1) * m
    one = z.copy()
    one[h // 2, w // 2] = m
    pairs = [("zero_max", z, f), ("max_zero", f, z), ("checker_inverse", chk, m - chk), ("checker_flat0", chk, z),
             ("checker_flatmax", chk, f), ("flat0_checker", z, chk), ("single", one, z)]
    return [(n, np.ascontiguousarray(a.astype(dt)), np.ascontiguousarray(b.astype(dt))) for n, a, b in pairs]


def weighted_sse_model(a, b, scale):
    """get_weighted_sse (dist.rs:234-283): per 4x4 chunk a u32 sum of squares, times its u32 scale
    in u64, rounded >> 8, summed in u64, then divided by 64 rounding to nearest"""
    h, w = a.shape
    total = 0
    for cy in range(h // 4):
        for cx in range(w // 4):
            d = a[4 * cy:4 * cy + 4, 4 * cx:4 * cx + 4].astype(np.int64) - b[4 * cy:4 * cy + 4, 4 * cx:4 * cx + 4]
            s = int((d * d).sum()) % U32
            total = (total + ((s * int(scale[cy, cx]) + 128) >> 8)) % U64
    return (total + 32) // 64


def ssim_boost_model(inp, svar, dvar, bd):
    """apply_ssim_boost (activity.rs:159-186, ssim_boost_rsqrt :107-143) in Python integers, with the
    u64 product wrapping (only an input near 2^32 with large variances reaches that).  Returns
    (result `as u32`, the value before that cast)."""
    cs = bd - 8
    sv, dv = svar >> (2 * cs), dvar >> (2 * cs)
    C1, C2, C3 = 3355, 16128, 12338
    ratio = (((C1 << 15) // C3) + 1) >> 1
    x = C1 * C1 + sv * dv
    k = (x.bit_length() - 1) >> 1
    s = 2 * k - 14
    t = (x >> s if s > 0 else x << -s) % (1 << 16)                 # `as u16`
    shift = 14 + ((s + 16) >> 1)
    n = t - 32768
    inner = -13490 + ((n * 6711) >> 15)
    norm = (23557 + ((n * inner) >> 15)) % (1 << 16)
    pre = ((inp * (((ratio * (sv + dv + C2)) * norm) >> 14)) % U64) >> shift     # u64 product
    return pre % U32, pre


AREA_DIVISORS = [round(16384 / n) for n in range(1, 65)]


def cdef_dist_model(a, b, bd):
    """cdef_dist_kernel (dist.rs:302-372): u32 sums wrapping, saturating variance subtraction,
    the 8x8-area scaling.  Returns (boosted `as u32`, before the cast, (svar, dvar, sse))."""
    s, d = a.astype(np.int64), b.astype(np.int64)
    sum_s, sum_d = int(s.sum()) % U32, int(d.sum()) % U32
    s2, d2, sd = int((s * s).sum()) % U32, int((d * d).sum()) % U32, int((s * d).sum()) % U32
    sse = (d2 + s2 - 2 * sd) % U32
    div = AREA_DIVISORS[s.size - 1]
    svar = max(s2 - (((sum_s * sum_s * div + 8192) >> 14) % U32), 0)
    dvar = max(d2 - (((sum_d * sum_d * div + 8192) >> 14) % U32), 0)
    svar = ((svar * div + 128) >> 8) % U32
    dvar = ((dvar * div + 128) >> 8) % U32
    boosted, pre = ssim_boost_model(sse, svar, dvar, bd)
    return boosted, pre, (svar, dvar, sse)


def variance_8x8_model(blk):
    """variance_8x8 (activity.rs:71-100): u16 column sums, u32 column sums of squares"""
    b = blk.astype(np.int64)
    cols = b.sum(0) % (1 << 16)
    s, s2 = int(cols.sum()), int((b * b).sum())
    v = s2 - ((s * s + 32) >> 6)
    return min(v, U32 - 1)


def activity_planes(bd):
    """all max, a 0/max checkerboard, 0/max stripes both ways, and unshifted noise (64 x 48)"""
    m = (1 << bd) - 1
    yy, xx = np.indices((48, 64))
    rng = np.random.default_rng(bd)
    return [np.ascontiguousarray(p.astype(pixel_dtype(bd))) for p in
            (np.full((48, 64), m), ((yy + xx) & 1) * m, (xx & 1) * m, (yy & 1) * m, rng.integers(0, m + 1, (48, 64)))]


@pytest.mark.parametrize("bd", BDS)
def test_weighted_sse_oracle_against_model(bd):
    """Oracle get_weighted_sse == weighted_sse_model on the full-contrast pairs, every size 4x4 ..
    128x128 (aspect <= 4), scales 1, 2^14 and 2^28 - 1 (and a mix of them)."""
    l = RL()
    fn = l.orc_weighted_sse_u8 if bd == 8 else l.orc_weighted_sse_u16
    rng = np.random.default_rng(bd)
    for w, h in WSSE_SIZES:
        mixed = rng.choice(SCALES, (h // 4, w // 4)).astype(np.uint32)
        for name, a, b in block_pairs(w, h, bd):
            for scale in [np.full((h // 4, w // 4), s, np.uint32) for s in SCALES] + [mixed]:
                got = fn(a.ctypes.data, w, b.ctypes.data, w, scale.ctypes.data, w // 4, w, h)
                assert got == weighted_sse_model(a, b, scale), (name, w, h, int(scale[0, 0]))
    m = (1 << bd) - 1
    a, b = block_pairs(128, 128, bd)[0][1:]
    big = np.full((32, 32), (1 << 28) - 1, np.uint32)
    assert fn(a.ctypes.data, 128, b.ctypes.data, 128, big.ctypes.data, 32, 128, 128) == \
        (((16 * m * m * ((1 << 28) - 1) + 128) >> 8) * 1024 + 32) // 64


CDEF_DIST_SIZES = [(w, h) for w in range(1, 9) for h in range(1, 9)]


@pytest.mark.parametrize("bd", BDS)
def test_cdef_dist_oracle_against_model(bd):
    """Oracle cdef_dist_kernel == cdef_dist_model (boosted value and the raw svar, dvar, sse) on the
    full-contrast pairs at every w x h up to 8x8.  At 12 bit the boosted value of a checkerboard
    against a flat block exceeds 2^32 before its final `as u32`: the result wraps, as in the
    reference."""
    l = RL()
    fn = l.orc_cdef_dist_kernel_u8 if bd == 8 else l.orc_cdef_dist_kernel_u16
    raw = (C.c_uint32 * 3)()
    wrapped = []
    for w, h in CDEF_DIST_SIZES:
        for name, a, b in block_pairs(8, 8, bd):
            got = fn(a.ctypes.data, 8, b.ctypes.data, 8, w, h, bd, raw)
            want, pre, want_raw = cdef_dist_model(a[:h, :w], b[:h, :w], bd)
            assert (got, tuple(raw)) == (want, want_raw), (name, w, h)
            assert got == l.orc_apply_ssim_boost(want_raw[2], want_raw[0], want_raw[1], bd)
            if pre >= U32:
                wrapped.append((name, w, h, pre))
    if bd == 12:
        print(f"\n12-bit cdef_dist: {len(wrapped)} cases wrap in apply_ssim_boost, largest pre-cast value "
              f"{max(p for *_, p in wrapped)}")
        assert ("checker_flat0", 8, 8, 45648943943) in wrapped
    else:
        assert not wrapped


@pytest.mark.parametrize("bd", BDS)
def test_ssim_boost_and_variance_models(bd):
    """apply_ssim_boost and variance_8x8 of the oracle == their Python models at the extremes: the
    activity mask's u16 column sums reach 8 * max (32760 at 12 bit) on all-max columns."""
    l = RL()
    l.orc_variance_8x8_u8.restype = l.orc_variance_8x8_u16.restype = C.c_uint32
    l.orc_variance_8x8_u8.argtypes = l.orc_variance_8x8_u16.argtypes = [C.c_void_p, C.c_ssize_t]
    var_fn = l.orc_variance_8x8_u8 if bd == 8 else l.orc_variance_8x8_u16
    m = (1 << bd) - 1
    top = 0
    for p in activity_planes(bd):
        for y in range(0, 48, 8):
            for x in range(0, 64, 8):
                blk = np.ascontiguousarray(p[y:y + 8, x:x + 8])
                v = var_fn(blk.ctypes.data, 8)
                assert v == variance_8x8_model(blk)
                assert l.orc_apply_ssim_boost(1 << 14, v, v, bd) == ssim_boost_model(1 << 14, v, v, bd)[0]
                top = max(top, int(blk.astype(np.int64).sum(0).max()))
    assert top == 8 * m
    for inp in (1, 1 << 14, U32 - 1):
        for sv in (0, 1, m * m * 16, (m * m * 64) >> 2, U32 - 1):
            for dv in (0, m * m * 16, U32 - 1):
                assert l.orc_apply_ssim_boost(inp, sv, dv, bd) == ssim_boost_model(inp, sv, dv, bd)[0], (inp, sv, dv)
