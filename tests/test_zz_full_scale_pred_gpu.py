"""GPU parity at full scale and at 12 bit for motion compensation, chroma-from-luma and the other
intra predictors, CDEF and the RDO distortions: CUDA (through the C ABI) == oracle, bit exact, on the
inputs of tests/test_full_scale_pred.py, which reach the i16 MC intermediate's table bounds, the i16
CfL samples at 32760, CDEF's direction search on unshifted high-bit-depth pixels and the u32 wrap of
the ssim-boosted distortion.  Where the CPU file has a Python model, the CUDA results are checked
against it as well."""
import ctypes as C

import numpy as np
import pytest

from rav1e_b200 import backend as B
from tests import gpu_util as G
from tests import oracle_lib as O
from tests.test_activity import oracle_mask
from tests.test_full_scale import pixel_dtype
from tests.test_full_scale_pred import (BDS, CDEF_DIST_SIZES, LAYOUTS, SCALES, U32, WSSE_SIZES, activity_planes,
                                        block_pairs, cdef_dist_model, cdef_planes, cfl_ac_inputs, cfl_ac_model,
                                        cfl_edges, cfl_lumas, cfl_pads, cfl_pred_model, h_only_tile, mc_avg_model,
                                        mc_fracs, mc_model, prep_bias, tap_sign_tile, taps, weighted_sse_model)
from tests.test_oracle_rdo_dist import L as RL
from tests.test_ref_abi_gpu import FILTERS

pytestmark = pytest.mark.gpu

M = {n: i for i, n in enumerate(O.MODES)}
vp, pd, i32 = C.c_void_p, C.c_ssize_t, C.c_int


def fn(name, restype=None):
    f = getattr(C.CDLL(B.LIB_PATH), name)
    f.restype = restype
    return f


def download(c, pl, like):
    out = np.zeros_like(like)
    c.check(c.L.b200_plane_download(c.h, C.byref(pl), out.ctypes.data, out.strides[0]))
    return out


# ---------------------------------------------------------------- 1. motion compensation

MC_SIZES = [(8, 8), (16, 16), (32, 32), (64, 64), (2, 2), (4, 4), (16, 8), (8, 32), (64, 16), (128, 128)]
MC_MODE_PAIRS = [(0, 0), (1, 1), (2, 2), (3, 3), (2, 0), (0, 1)]
TILE_KINDS = 3          # tap-sign tile of sign +1, of sign -1, H-only pattern of sign +1


def mc_mosaic(w, h, bd, mx, my, dec):
    """A plane of (h+8) x (w+8) cells, each holding the footprint of one block: the tile of
    TILE_KINDS for its fraction pair.  Returns (plane image, blocks, mvs, [(cf, rf, kind, fx, fy)]).
    The vector of a block lands its footprint on its own cell: the integer part is 0, the fraction
    is the cell's (luma vectors address only even fractions)."""
    fracs = mc_fracs(1 if dec else 2)
    cells = [(cf, rf, k) for cf, rf in fracs for k in range(TILE_KINDS)]
    ncol = 16
    cw, ch = w + 8, h + 8
    nrow = -(-len(cells) // ncol)
    img = np.zeros((nrow * ch, ncol * cw), pixel_dtype(bd))
    blocks = np.zeros(len(cells), B.BLOCK_DTYPE)
    mvs = np.zeros((len(cells), 2), np.int16)
    meta = []
    for i, (cf, rf, k) in enumerate(cells):
        fx, fy = taps(mx, cf, w), taps(my, rf, h)
        tile = h_only_tile(fx, w, h, bd, 1) if k == 2 else tap_sign_tile(fx, fy, w, h, bd, 1 if k == 0 else -1)
        x0, y0 = (i % ncol) * cw, (i // ncol) * ch
        img[y0:y0 + h + 7, x0:x0 + w + 7] = tile
        blocks[i] = (x0 + 3, y0 + 3)
        mvs[i] = (rf, cf) if dec else (rf // 2, cf // 2)
        meta.append((cf, rf, k, fx, fy, tile))
    return img, blocks, mvs, meta


@pytest.mark.parametrize("bd", BDS)
@pytest.mark.parametrize("w,h", MC_SIZES)
def test_mc_blocks_on_tap_sign_tiles(w, h, bd):
    """b200_mc_blocks_dev put (the packed fast kernel for the squares 8..64 at 4:4:4, the generic one
    otherwise) and prep, luma and 4:2:0 chroma vectors, six mode pairs covering all four modes in each
    direction: == oracle and == the int64 model.  b200_mc_avg_dev on the extreme preps in both sign
    combinations == oracle and model."""
    import torch
    c = G.ctx()
    tdt = torch.uint8 if bd == 8 else torch.int16
    for mx, my in MC_MODE_PAIRS:
        for dec in (0, 1):
            img, blocks, mvs, meta = mc_mosaic(w, h, bd, mx, my, dec)
            n = len(blocks)
            op, dp = G.both_planes(img, 8)
            d_blocks, d_mvs = G.to_dev(blocks), G.to_dev(mvs)
            outs = []
            for kind in (0, 1):
                want = O.mc_blocks(op, blocks, mvs, w, h, mx, my, bd, dec, dec, kind)
                d_out = torch.empty((n, h, w), dtype=tdt if kind == 0 else torch.int16, device="cuda")
                c.mc_blocks_dev(dp, d_blocks, d_mvs, n, w, h, mx, my, bd, dec, dec, kind, d_out)
                c.synchronize()
                got = d_out.cpu().numpy().view(want.dtype)
                msg = f"modes {mx}{my} dec {dec} kind {kind}"
                np.testing.assert_array_equal(got, want, err_msg=msg)
                outs.append(got)
            for i, (cf, rf, k, fx, fy, tile) in enumerate(meta):
                put, pre, _ = mc_model(tile, fx, fy, w, h, bd)
                np.testing.assert_array_equal(outs[0][i], put, err_msg=f"modes {mx}{my} frac {cf},{rf} kind {k}")
                np.testing.assert_array_equal(outs[1][i], pre - prep_bias(bd), err_msg=f"modes {mx}{my} frac {cf},{rf}")
            plus = np.array([i for i, m in enumerate(meta) if m[2] == 0])
            minus = np.array([i for i, m in enumerate(meta) if m[2] == 1])
            for a, b in ((plus, plus), (plus, minus), (minus, minus), (minus, plus)):
                t1, t2 = np.ascontiguousarray(outs[1][a]), np.ascontiguousarray(outs[1][b])
                d_dst = torch.empty((len(a), h, w), dtype=tdt, device="cuda")
                c.mc_avg_dev(torch.from_numpy(t1).cuda(), torch.from_numpy(t2).cuda(), d_dst, len(a), w, h, bd)
                c.synchronize()
                got = d_dst.cpu().numpy().view(pixel_dtype(bd))
                want = np.stack([O.mc_avg(x, y, bd) for x, y in zip(t1, t2)])
                np.testing.assert_array_equal(got, want)
                np.testing.assert_array_equal(got, mc_avg_model(t1, t2, bd))
            c.plane_free(dp)


PERCALL_FRACS = [(0, 0), (5, 0), (0, 11), (7, 13), (15, 1), (8, 8)]


@pytest.mark.parametrize("bd", BDS)
def test_mc_percall_symbols_on_tap_sign_tiles(bd):
    """b200_put_8tap / b200_prep_8tap / b200_mc_avg for all 16 mode pairs, and at 10/12 bit the
    reference-signature rav1e_put_* / rav1e_prep_* / rav1e_avg_16bpc_cuda with bitdepth_max, on the
    tap-sign tiles of both signs."""
    L = B.lib()
    isz = np.dtype(pixel_dtype(bd)).itemsize
    hbd = [(1 << bd) - 1] if bd > 8 else []
    bpc = 8 if bd == 8 else 16
    pairs = [(f"{mx}{my}", mx, my, None) for mx in range(4) for my in range(4)]
    pairs += [(name, mx, my, name) for name, mx, my in FILTERS]
    for w, h in ((8, 8), (16, 8), (4, 4)):
        for label, mx, my, name in pairs:
            if name:
                put, prep = fn(f"rav1e_put_{name}_{bpc}bpc_cuda"), fn(f"rav1e_prep_{name}_{bpc}bpc_cuda")
                put.argtypes = [vp, pd, vp, pd, i32, i32, i32, i32] + [i32] * len(hbd)
                prep.argtypes = [vp, vp, pd, i32, i32, i32, i32] + [i32] * len(hbd)
            for cf, rf in PERCALL_FRACS:
                fx, fy = taps(mx, cf, w), taps(my, rf, h)
                preps = []
                for sign in (1, -1):
                    tile = tap_sign_tile(fx, fy, w, h, bd, sign)
                    op = O.Plane(w + 7, h + 7, 0, tile.dtype)
                    op.fill_from(tile)
                    src, st = op.at(3, 3), op.stride * isz
                    want = O.put_8tap(op, 3, 3, w, h, cf, rf, mx, my, bd)
                    wantp = O.prep_8tap(op, 3, 3, w, h, cf, rf, mx, my, bd)
                    got, gotp = np.zeros((h, w), tile.dtype), np.zeros((h, w), np.int16)
                    if name:
                        put(got.ctypes.data, w * isz, src, st, w, h, cf, rf, *hbd)
                        prep(gotp.ctypes.data, src, st, w, h, cf, rf, *hbd)
                    else:
                        L.b200_put_8tap(got.ctypes.data, w * isz, src, st, w, h, cf, rf, mx, my, bd)
                        L.b200_prep_8tap(gotp.ctypes.data, src, st, w, h, cf, rf, mx, my, bd)
                    msg = f"{label} {w}x{h} frac {cf},{rf} sign {sign}"
                    np.testing.assert_array_equal(got, want, err_msg=msg)
                    np.testing.assert_array_equal(gotp, wantp, err_msg=msg)
                    preps.append(wantp)
                for t1, t2 in ((preps[0], preps[1]), (preps[0], preps[0]), (preps[1], preps[1])):
                    got = np.zeros((h, w), pixel_dtype(bd))
                    if name and bd > 8:
                        avg = fn(f"rav1e_avg_{bpc}bpc_cuda")
                        avg.argtypes = [vp, pd, vp, vp, i32, i32, i32]
                        avg(got.ctypes.data, w * isz, t1.ctypes.data, t2.ctypes.data, w, h, *hbd)
                    else:
                        L.b200_mc_avg(got.ctypes.data, w * isz, t1.ctypes.data, t2.ctypes.data, w, h, bd)
                    np.testing.assert_array_equal(got, O.mc_avg(t1, t2, bd))


# ---------------------------------------------------------------- 2. chroma from luma and intra prediction

CFL_CASES = [(4, 4), (8, 8), (16, 16), (32, 32), (16, 8), (8, 32)]


@pytest.mark.parametrize("bd", BDS)
@pytest.mark.parametrize("xdec,ydec", LAYOUTS)
def test_cfl_ac_full_scale(xdec, ydec, bd):
    """b200_pred_cfl_ac_dev on the full-scale lumas, every valid w_pad / h_pad: == oracle, == the
    model; at 12 bit the samples reach 32760."""
    import torch
    c = G.ctx()
    for bw, bh in CFL_CASES:
        lw, lh = bw << xdec, bh << ydec
        lumas = cfl_lumas(lw, lh, bd, xdec, ydec)
        img = np.ascontiguousarray(np.concatenate(lumas, axis=1))
        pl = c.plane_from_host(img, 0)
        n = len(lumas)
        blocks = np.zeros(n, B.BLOCK_DTYPE)
        blocks["x"] = np.arange(n) * lw
        d_blocks = G.to_dev(blocks)
        for w_pad, h_pad in cfl_pads(bw, bh, xdec, ydec):
            d_ac = torch.empty((n, bw * bh), dtype=torch.int16, device="cuda")
            c.pred_cfl_ac_dev(pl, d_blocks, n, bw, bh, w_pad, h_pad, xdec, ydec, d_ac)
            c.synchronize()
            got = d_ac.cpu().numpy()
            for i, luma in enumerate(lumas):
                msg = f"{bw}x{bh} pad {w_pad}{h_pad} luma {i}"
                np.testing.assert_array_equal(got[i], O.pred_cfl_ac(luma, bw, bh, w_pad, h_pad, xdec, ydec), err_msg=msg)
                want, s = cfl_ac_model(luma, bw, bh, w_pad, h_pad, xdec, ydec)
                np.testing.assert_array_equal(got[i], want, err_msg=msg)
                if bd == 12 and i == 0:
                    assert (s == 32760).all()
        c.plane_free(pl)


def run_items(edges, items, w, h, bd, ac=None):
    import torch
    c = G.ctx()
    n = len(items)
    d_out = torch.empty((n, h, w), dtype=torch.uint8 if bd == 8 else torch.int16, device="cuda")
    c.predict_intra_dev(G.to_dev(edges), G.to_dev(items), n, None if ac is None else G.to_dev(ac), w, h, bd,
                        4096, 4096, d_out)
    c.synchronize()
    return d_out.cpu().numpy().view(edges.dtype)


def test_cfl_prediction_12bit_every_alpha():
    """b200_predict_intra_dev UV_CFL_PRED at 12 bit: every alpha in -16..16, all four DC variants, edges
    at 0, at max and mixed, extreme ac blocks: == oracle and == the model (the clip at 4095 engages)."""
    bd = 12
    edges = np.stack(cfl_edges(bd))
    by_size = {}
    for bw, bh, ac in cfl_ac_inputs(bd):
        by_size.setdefault((bw, bh), []).append(ac)
    for (bw, bh), acs in by_size.items():
        rows = [(ei, ai, variant, alpha) for ei in range(len(edges)) for ai in range(len(acs))
                for variant in range(4) for alpha in range(-16, 17)]
        items = np.zeros(len(rows), B.INTRA_ITEM_DTYPE)
        for k, (ei, ai, variant, alpha) in enumerate(rows):
            items[k] = (ei, ai, 64, 64, alpha, M["UV_CFL_PRED"], variant, -1, bh, bw, 0)
        ac_all = np.ascontiguousarray(np.stack(acs))
        got = run_items(edges, items, bw, bh, bd, ac=ac_all)
        for k, (ei, ai, variant, alpha) in enumerate(rows):
            want = O.predict_intra(M["UV_CFL_PRED"], variant, edges[ei], bw, bh, bd, angle=alpha, ac=acs[ai],
                                   left_len=bh, above_len=bw)
            msg = f"{bw}x{bh} edge {ei} ac {ai} var {variant} alpha {alpha}"
            np.testing.assert_array_equal(got[k], want, err_msg=msg)
            np.testing.assert_array_equal(got[k], cfl_pred_model(edges[ei], variant, acs[ai], alpha, bw, bh, bd),
                                          err_msg=msg)
        assert (got == 4095).any() and (got == 0).any()


def intra_edges_12bit():
    """0/max alternating (period 1 and 2), step edges (above max / left 0 and the reverse, and a step
    in the middle of the above edge), all max"""
    m = 4095
    i = np.arange(O.EDGE_LEN)
    e = [(i & 1) * m, ((i >> 1) & 1) * m, np.where(i > 128, m, 0), np.where(i < 128, m, 0),
         np.where(i > 136, m, 0), np.full(O.EDGE_LEN, m)]
    return np.ascontiguousarray(np.stack(e).astype(np.uint16))


def test_intra_modes_12bit_full_contrast_edges():
    """Directional (with edge filter and upsampling), smooth and Paeth modes at 12 bit on 0/max
    alternating and step edges, every TxSize: == oracle; the filters' overshoot hits the clip."""
    bd = 12
    edges = intra_edges_12bit()
    for w, h in O.TX_SIZES:
        full = min(128, w + h)
        rows = []
        for ei in range(len(edges)):
            for mode in ("SMOOTH_PRED", "SMOOTH_V_PRED", "SMOOTH_H_PRED", "PAETH_PRED"):
                rows.append((ei, M[mode], 3, 0, -1, h, w))
            for mode, base in O.MODE_ANGLE.items():
                for delta in (-3, 0, 3):
                    for ief in (-1, 0, 1):
                        rows.append((ei, M[mode], 3, base + 3 * delta, ief, full, full))
        items = np.zeros(len(rows), B.INTRA_ITEM_DTYPE)
        for k, (ei, mode, variant, angle, ief, ll, al) in enumerate(rows):
            items[k] = (ei, 0, 64, 64, angle, mode, variant, ief, ll, al, 0)
        got = run_items(edges, items, w, h, bd)
        for k, (ei, mode, variant, angle, ief, ll, al) in enumerate(rows):
            want = O.predict_intra(mode, variant, edges[ei], w, h, bd, angle=angle, ief=ief, left_len=ll, above_len=al)
            np.testing.assert_array_equal(got[k], want, err_msg=f"{w}x{h} {O.MODES[mode]} angle {angle} ief {ief} "
                                          f"edge {ei}")


def test_cfl_percall_symbols_12bit():
    """rav1e_ipred_cfl_ac_{420,422,444}_16bpc_cuda and rav1e_ipred_cfl[_128|_left|_top]_16bpc_cuda with
    bitdepth_max 4095 on the full-scale lumas and edges, alphas -16, -1, 1, 16."""
    bd, bdmax = 12, 4095
    edges = cfl_edges(bd)
    for lay, xdec, ydec in (("420", 1, 1), ("422", 1, 0), ("444", 0, 0)):
        fac = fn(f"rav1e_ipred_cfl_ac_{lay}_16bpc_cuda")
        fac.argtypes = [vp, vp, pd, i32, i32, i32, i32]
        for bw, bh, w_pad, h_pad in ((8, 8, 0, 0), (16, 16, 1, 2), (32, 32, 3, 3), (16, 8, 0, 1)):
            for luma in cfl_lumas(bw << xdec, bh << ydec, bd, xdec, ydec):
                ac = np.zeros(bw * bh, np.int16)
                fac(ac.ctypes.data, luma.ctypes.data, luma.strides[0], w_pad, h_pad, bw, bh)
                np.testing.assert_array_equal(ac, O.pred_cfl_ac(luma, bw, bh, w_pad, h_pad, xdec, ydec))
                for edge in edges:
                    topleft = edge.ctypes.data + 128 * 2
                    for name, variant in (("cfl", 3), ("cfl_128", 0), ("cfl_left", 1), ("cfl_top", 2)):
                        f = fn(f"rav1e_ipred_{name}_16bpc_cuda")
                        f.argtypes = [vp, pd, vp, i32, i32, vp, i32, i32]
                        for alpha in (-16, -1, 1, 16):
                            got = np.zeros((bh, bw), np.uint16)
                            f(got.ctypes.data, bw * 2, topleft, bw, bh, ac.ctypes.data, alpha, bdmax)
                            want = O.predict_intra(M["UV_CFL_PRED"], variant, edge, bw, bh, bd, angle=alpha, ac=ac,
                                                   left_len=bh, above_len=bw)
                            np.testing.assert_array_equal(got, want, err_msg=f"{name} {lay} {bw}x{bh} {alpha}")


# ---------------------------------------------------------------- 3. CDEF

CDEF_W, CDEF_H = 9 * 64 - 40, 8 * 64 - 24        # 9 x 8 = 72 superblocks, partial at the right and bottom


@pytest.mark.parametrize("bd", [10, 12])
def test_cdef_direction_unshifted(bd):
    """b200_cdef_find_dir_dev, b200_cdef_dir and rav1e_cdef_dir_16bpc_cuda on unshifted noise and the
    full-contrast planes: == oracle, and == the 8-bit search of the top 8 bits."""
    import torch
    c = G.ctx()
    L = B.lib()
    fdir = fn("rav1e_cdef_dir_16bpc_cuda", i32)
    fdir.argtypes = [vp, pd, C.POINTER(C.c_uint32), i32]
    W, H = 128, 64
    for name, img in cdef_planes(W, H, bd, seed=bd).items():
        dirs, var = O.cdef_analyze_frame(img, bd)
        d8, v8 = O.cdef_analyze_frame(np.ascontiguousarray((img >> (bd - 8)).astype(np.uint8)), 8)
        np.testing.assert_array_equal(dirs, d8, err_msg=name)
        np.testing.assert_array_equal(var, v8, err_msg=name)
        pl = c.plane_from_host(img, 0)
        d_dir = torch.empty(dirs.size, dtype=torch.uint8, device="cuda")
        d_var = torch.empty(var.size, dtype=torch.int32, device="cuda")
        c.cdef_find_dir_dev(pl, bd, None, d_dir, d_var)
        c.synchronize()
        np.testing.assert_array_equal(d_dir.cpu().numpy().reshape(dirs.shape), dirs, err_msg=name)
        np.testing.assert_array_equal(d_var.cpu().numpy().reshape(var.shape), var, err_msg=name)
        c.plane_free(pl)
        for by, bx in ((0, 0), (3, 7), (7, 15), (4, 2)):
            blk = img[8 * by:8 * by + 8, 8 * bx:8 * bx + 8]
            want = O.cdef_find_dir(np.ascontiguousarray(blk), bd)
            v = C.c_uint32()
            p = img.ctypes.data + (8 * by * W + 8 * bx) * 2
            assert (L.b200_cdef_dir(p, W * 2, C.byref(v), bd), v.value) == want, (name, by, bx)
            assert (fdir(p, W * 2, C.byref(v), (1 << bd) - 1), v.value) == want, (name, by, bx)


def cdef_frame_inputs(bd, xdec, ydec, seed):
    """(name, luma, chroma) on the CDEF_W x CDEF_H frame for every cdef_planes pattern"""
    lum = cdef_planes(CDEF_W, CDEF_H, bd, seed)
    chr_ = cdef_planes(CDEF_W >> xdec, CDEF_H >> ydec, bd, seed + 1)
    return [(k, lum[k], chr_[k]) for k in lum]


@pytest.mark.parametrize("bd", [10, 12])
@pytest.mark.parametrize("xdec,ydec", LAYOUTS)
def test_cdef_frame_all_strengths(bd, xdec, ydec):
    """b200_cdef_filter_plane_dev (luma and chroma) on every full-scale pattern, all 64 strength codes
    (one per superblock), damping 3 and 6, a skip mask: == oracle; b200_cdef_filter_rect_dev per
    64x64-aligned tile and b200_cdef_tiles_dev == the whole-frame result."""
    import torch
    c = G.ctx()
    rng = np.random.default_rng(bd * 10 + xdec * 2 + ydec)
    W, H = CDEF_W, CDEF_H
    sbw, sbh = (W + 63) // 64, (H + 63) // 64
    assert sbw * sbh >= 64
    codes = (np.arange(sbw * sbh) % 64).astype(np.uint8)
    y_str = np.ascontiguousarray(codes.reshape(sbh, sbw))
    uv_str = np.ascontiguousarray(rng.permutation(codes).reshape(sbh, sbw))
    skip8 = (rng.random((H // 8, W // 8)) < 0.15).astype(np.uint8)
    d_skip = G.to_dev(skip8)
    n8 = (H // 8) * (W // 8)
    # three superblock-aligned tiles covering the frame, in 8x8 luma blocks (the last ones partial)
    w8, h8 = W // 8, H // 8
    rects = [(0, 0, 32, h8), (32, 0, w8 - 32, 24), (32, 24, w8 - 32, h8 - 24)]
    for name, luma, chroma in cdef_frame_inputs(bd, xdec, ydec, seed=bd + xdec):
        dirs, var = O.cdef_analyze_frame(luma, bd, skip8)
        pl_y = c.plane_from_host(luma, 0)
        d_dir = torch.empty(n8, dtype=torch.uint8, device="cuda")
        d_var = torch.empty(n8, dtype=torch.int32, device="cuda")
        c.cdef_find_dir_dev(pl_y, bd, d_skip, d_dir, d_var)
        c.synchronize()
        np.testing.assert_array_equal(d_dir.cpu().numpy().reshape(dirs.shape), dirs, err_msg=name)
        np.testing.assert_array_equal(d_var.cpu().numpy().reshape(var.shape), var, err_msg=name)
        for damping in (3, 6):
            for img, plane, xd, yd, strn in ((luma, 0, 0, 0, y_str), (chroma, 1, xdec, ydec, uv_str)):
                want = O.cdef_filter_plane(img, plane, xd, yd, W, H, bd, damping, skip8, dirs, var, strn)
                msg = f"{name} plane {plane} damping {damping}"
                pin = pl_y if plane == 0 else c.plane_from_host(img, 0)
                d_str = G.to_dev(strn)
                outs = [c.plane_from_host(np.zeros_like(img), 0) for _ in range(3)]
                c.cdef_filter_plane_dev(pin, outs[0], plane, xd, yd, W, H, bd, damping, d_skip, d_dir, d_var, d_str)
                items = (B.CdefItem * len(rects))()
                for k, r8 in enumerate(rects):
                    c.cdef_filter_rect_dev(pin, outs[1], plane, xd, yd, W, H, bd, damping, d_skip, d_dir, d_var,
                                           d_str, r8)
                    it = items[k]
                    it.inp, it.out = C.pointer(pin), C.pointer(outs[2])
                    it.d_skip8, it.d_dir, it.d_var = d_skip.data_ptr(), d_dir.data_ptr(), d_var.data_ptr()
                    it.rx8, it.ry8, it.rw8, it.rh8 = r8
                c.cdef_tiles_dev(items, plane, xd, yd, W, H, bd, damping, d_str, find_dir=False)
                c.synchronize()
                for k, o in enumerate(outs):
                    np.testing.assert_array_equal(download(c, o, img), want, err_msg=f"{msg} path {k}")
                    c.plane_free(o)
                if plane:
                    c.plane_free(pin)
        c.plane_free(pl_y)


# ---------------------------------------------------------------- 4. RDO distortions

def side_by_side(pairs):
    a = np.ascontiguousarray(np.concatenate([p[1] for p in pairs], axis=1))
    b = np.ascontiguousarray(np.concatenate([p[2] for p in pairs], axis=1))
    return a, b


@pytest.mark.parametrize("bd", BDS)
def test_weighted_sse_full_contrast(bd):
    """b200_weighted_sse_dev on the full-contrast pairs at every size 4x4 .. 128x128, scales 1, 2^14,
    2^28 - 1 and a mix: == oracle and == the Python model; b200_weighted_sse at 128x128."""
    c = G.ctx()
    ol = RL()
    ofn = ol.orc_weighted_sse_u8 if bd == 8 else ol.orc_weighted_sse_u16
    rng = np.random.default_rng(bd)
    for w, h in WSSE_SIZES:
        pairs = block_pairs(w, h, bd)
        a, b = side_by_side(pairs)
        W = a.shape[1]
        da, db = c.plane_from_host(a, 0), c.plane_from_host(b, 0)
        n = len(pairs)
        blocks = np.zeros(n, B.BLOCK_DTYPE)
        blocks["x"] = np.arange(n) * w
        d_blocks = G.to_dev(blocks)
        for scale in [np.full((h // 4, W // 4), s, np.uint32) for s in SCALES] + \
                [rng.choice(SCALES, (h // 4, W // 4)).astype(np.uint32)]:
            d_out = G.dev_empty(8 * n)
            c.weighted_sse_dev(da, db, d_blocks, n, w, h, G.to_dev(scale), W // 4, d_out)
            c.synchronize()
            got = G.from_dev(d_out, np.uint64)[:n]
            for i, (name, pa, pb) in enumerate(pairs):
                sc = np.ascontiguousarray(scale[:, i * w // 4:(i + 1) * w // 4])
                want = ofn(pa.ctypes.data, w, pb.ctypes.data, w, sc.ctypes.data, w // 4, w, h)
                assert int(got[i]) == want == weighted_sse_model(pa, pb, sc), (name, w, h, int(sc[0, 0]))
                if (w, h) == (128, 128) and i < 2:
                    pc = B.lib().b200_weighted_sse(pa.ctypes.data, w * pa.itemsize, pb.ctypes.data, w * pb.itemsize,
                                                   sc.ctypes.data, (w // 4) * 4, w, h, pa.itemsize)
                    assert pc == want, (name, int(sc[0, 0]))
        c.plane_free(da)
        c.plane_free(db)


@pytest.mark.parametrize("bd", BDS)
def test_cdef_dist_full_contrast(bd):
    """b200_cdef_dist_dev (boosted and raw outputs) on the full-contrast 8x8 pairs at every w x h up to
    8x8, and b200_cdef_dist_kernel: == oracle and == the Python model, including the 12-bit cases whose
    boosted value wraps modulo 2^32."""
    c = G.ctx()
    ol = RL()
    ofn = ol.orc_cdef_dist_kernel_u8 if bd == 8 else ol.orc_cdef_dist_kernel_u16
    pairs = block_pairs(8, 8, bd)
    a, b = side_by_side(pairs)
    da, db = c.plane_from_host(a, 0), c.plane_from_host(b, 0)
    n = len(pairs)
    blocks = np.zeros(n, B.BLOCK_DTYPE)
    blocks["x"] = np.arange(n) * 8
    d_blocks = G.to_dev(blocks)
    r3, g3 = (C.c_uint32 * 3)(), (C.c_uint32 * 3)()
    wrapped = 0
    for w, h in CDEF_DIST_SIZES:
        d_out, d_raw = G.dev_empty(4 * n), G.dev_empty(12 * n)
        c.cdef_dist_dev(da, db, d_blocks, n, w, h, bd, d_out, d_raw)
        c.synchronize()
        got, raw = G.from_dev(d_out, np.uint32)[:n], G.from_dev(d_raw, np.uint32)[:3 * n].reshape(n, 3)
        for i, (name, pa, pb) in enumerate(pairs):
            want = ofn(pa.ctypes.data, 8, pb.ctypes.data, 8, w, h, bd, r3)
            model, pre, model_raw = cdef_dist_model(pa[:h, :w], pb[:h, :w], bd)
            assert int(got[i]) == want == model, (name, w, h)
            assert tuple(int(v) for v in raw[i]) == tuple(r3) == model_raw, (name, w, h)
            wrapped += pre >= U32
            if (w, h) in ((8, 8), (4, 4), (8, 3)):
                pc = B.lib().b200_cdef_dist_kernel(pa.ctypes.data, 8 * pa.itemsize, pb.ctypes.data, 8 * pb.itemsize,
                                                   w, h, bd, g3)
                assert pc == want and tuple(g3) == tuple(r3), (name, w, h)
    assert (wrapped > 0) == (bd == 12)
    c.plane_free(da)
    c.plane_free(db)


def test_activity_mask_12bit_full_scale():
    """b200_activity_mask_dev at 12 bit on all-max, checkerboard, stripe and noise planes (u16 column
    sums at 32760): == oracle."""
    c = G.ctx()
    for k, img in enumerate(activity_planes(12)):
        var, sc, _ = oracle_mask(img, 16, 12)
        dpl = c.plane_from_host(img, 16)
        n = var.size
        d_var, d_sc = G.dev_empty(4 * n), G.dev_empty(4 * n)
        c.activity_mask_dev(dpl, 12, d_var, d_sc)
        c.synchronize()
        np.testing.assert_array_equal(G.from_dev(d_var, np.uint32)[:n].reshape(var.shape), var, err_msg=str(k))
        np.testing.assert_array_equal(G.from_dev(d_sc, np.uint32)[:n].reshape(sc.shape), sc, err_msg=str(k))
        c.plane_free(dpl)
