"""GPU parity at full scale and at 12 bit: CUDA (through the C ABI) == oracle, bit exact, on the
inputs of tests/test_full_scale.py, which reach the limits the kernels' integer arithmetic is built
around: the packed u16 lanes of the HBD SAD (8 rows x 4095 < 2^16), the i16 MC intermediate, the
forward transform's output cast, the quantizer's wrapping i32 products, and the inverse transform's
row clamp, rectangular scaling product, column clamp and pixel clip.  Where a cheap independent
model exists (SAD of a constant difference, the Hadamard SATD, the float transform) the CUDA
results are checked against it as well."""
import numpy as np
import pytest

from rav1e_b200 import backend as B
from tests import gpu_util as G
from tests import oracle_lib as O
from tests.test_full_scale import (BDS, PATTERNS, SCAN_TYPES, STEPS, assert_near_float_model, coeff_dtype,
                                   full_scale_planes, fwd_extreme_inputs, hadamard_satd, inverse_inputs,
                                   inverse_reference, pixel_dtype, quant_inputs, side_by_side_blocks)
from tests.test_me_gpu import CAND_CASES
from tests.test_me_search_gpu import predictor_subsets
from tests.test_oracle_inv_txfm import inverse_add
from tests.test_oracle_quantize import L as OL
from tests.test_oracle_quantize import chain as oracle_chain
from tests.test_quantize_gpu import run_gpu as quantize_gpu
from tests.test_zz_inv_txfm_gpu import download

pytestmark = pytest.mark.gpu

EMPTY = np.uint64(2**64 - 1)
LAM = 20000        # large enough that the rate term, not the SAD, separates tied candidates


def planes(pattern, W, H, PAD, bd, seed):
    cur, ref = full_scale_planes(pattern, W, H, bd, seed=seed)
    ocur, dcur = G.both_planes(cur, PAD)
    oref, dref = G.both_planes(ref, PAD)
    return cur, ref, ocur, dcur, oref, dref


def free(*pls):
    for p in pls:
        G.ctx().plane_free(p)


def check_winners(best, want_sad, want_cost, cands, offs):
    """per block: the first candidate of least cost (EMPTY when none is in range)"""
    nb = len(offs) - 1
    order = np.lexsort((np.arange(len(cands)), want_cost, cands["block"]))
    for b in range(nb):
        lo, hi = int(offs[b]), int(offs[b + 1])
        if lo == hi or want_cost[order[lo]] == EMPTY:
            assert best[b]["cost"] == EMPTY, b
            continue
        k = order[lo]
        assert best[b]["cost"] == want_cost[k] and best[b]["sad"] == want_sad[k], b
        assert (best[b]["mv_row"], best[b]["mv_col"]) == (cands[k]["mv_row"], cands[k]["mv_col"]), b


# ---------------------------------------------------------------- 1. distortion and ME at full contrast

@pytest.mark.parametrize("bd", BDS)
def test_percall_symbols_full_contrast(bd):
    """rav1e_sad*/satd*_cuda and the _hbd forms, every block size, at two offsets (the checkerboard's
    phase flips at the odd one): == oracle, == the numpy Hadamard model, and SAD == w*h*max on the
    constant patterns."""
    L = B.lib()
    OLIB = O.lib()
    hbd = bd > 8
    maxv = (1 << bd) - 1
    for pattern in PATTERNS:
        cur, ref = full_scale_planes(pattern, 160, 144, bd, seed=bd)
        st = cur.shape[1]
        isz = cur.itemsize
        for w, h in B.BLOCK_SIZES:
            for x0, y0 in ((0, 0), (5, 3)):
                a, b = cur[y0:y0 + h, x0:x0 + w], ref[y0:y0 + h, x0:x0 + w]
                pa, pb = O.ptr(cur, y0 * st + x0), O.ptr(ref, y0 * st + x0)
                sad_o = (OLIB.orc_get_sad_u16 if hbd else OLIB.orc_get_sad_u8)(pa, st, pb, st, w, h)
                satd_o = (OLIB.orc_get_satd_u16 if hbd else OLIB.orc_get_satd_u8)(pa, st, pb, st, w, h)
                if hbd:
                    sad = getattr(L, f"rav1e_sad_{w}x{h}_hbd_cuda")(pa, st * isz, pb, st * isz)
                    satd = getattr(L, f"rav1e_satd_{w}x{h}_hbd_cuda")(pa, st * isz, pb, st * isz, maxv)
                else:
                    sad = getattr(L, f"rav1e_sad{w}x{h}_cuda")(pa, st, pb, st)
                    satd = getattr(L, f"rav1e_satd_{w}x{h}_cuda")(pa, st, pb, st)
                ctx = (pattern, w, h, x0)
                assert sad == sad_o == int(np.abs(a.astype(np.int64) - b).sum()), ctx
                assert satd == satd_o == hadamard_satd(a, b), ctx
                if pattern in ("max_vs_zero", "zero_vs_max"):
                    assert sad == w * h * maxv
        # the generic path for non-canonical crops
        for w, h in ((16, 12), (12, 8), (20, 20)):
            pa, pb = O.ptr(cur), O.ptr(ref)
            want = (OLIB.orc_get_sad_u16 if hbd else OLIB.orc_get_sad_u8)(pa, st, pb, st, w, h)
            assert L.b200_get_sad(pa, st * isz, pb, st * isz, w, h, isz) == want
            want = (OLIB.orc_get_satd_u16 if hbd else OLIB.orc_get_satd_u8)(pa, st, pb, st, w, h)
            assert L.b200_get_satd(pa, st * isz, pb, st * isz, w, h, isz) == want


CAND_SIZES = sorted({(w, h) for w, h, *_ in CAND_CASES})
# (per_block, max_px, window_hint_px): dense lists (grouped kernel) with a 16-aligned and an unaligned
# hint, and sparse lists (the chunk-list kernel)
LISTS = [(40, 32, 32), (44, 20, 20), (3, 40, 40), (2, 60, 60)]


@pytest.mark.parametrize("bd", BDS)
@pytest.mark.parametrize("w,h", CAND_SIZES)
def test_candidate_lists_full_contrast(w, h, bd):
    W, H, PAD = 256, 128, 160
    c = G.ctx()
    dtype = pixel_dtype(bd)
    blocks = G.grid_blocks(W, H, w, h)
    nb = len(blocks)
    rng = np.random.default_rng(w * 131 + h + bd)
    pmv = (rng.integers(-64, 65, (nb, 4)) * 4).astype(np.int16)
    d_blocks, d_pmv = G.to_dev(blocks), G.to_dev(pmv)
    for k, pattern in enumerate(PATTERNS):
        cur, ref, ocur, dcur, oref, dref = planes(pattern, W, H, PAD, bd, seed=w + h + k)
        assert cur.dtype == dtype
        for per_block, max_px, hint in LISTS:
            cands, offs = G.random_cands(nb, per_block, max_px, seed=7 + k, fullpel=(w != 8))
            n = len(cands)
            for use_satd in (False, True):
                want_sad, want_cost = O.fullpel_candidates(ocur, oref, blocks, cands, w, h, use_satd, LAM, pmv)
                p = B.me_params(w, h, W, H, LAM, use_satd=use_satd, bit_depth=bd, window_hint_px=hint)
                d_sad, d_cost, d_best = G.dev_empty(4 * n), G.dev_empty(8 * n), G.dev_empty(16 * nb)
                c.me_candidates_dev(dcur, dref, d_blocks, nb, G.to_dev(cands), n, p, G.to_dev(offs), d_pmv,
                                    d_sad, d_cost, d_best)
                # ungrouped call (no CSR offsets): per-candidate outputs only
                perm = np.random.default_rng(1).permutation(n)
                d_sad2 = G.dev_empty(4 * n)
                c.me_candidates_dev(dcur, dref, d_blocks, nb, G.to_dev(cands[perm]), n, p, None, d_pmv, d_sad2,
                                    None, None)
                c.synchronize()
                msg = f"{pattern} list={per_block} satd={use_satd}"
                np.testing.assert_array_equal(G.from_dev(d_sad, np.uint32)[:n], want_sad, err_msg=msg)
                np.testing.assert_array_equal(G.from_dev(d_cost, np.uint64)[:n], want_cost, err_msg=msg)
                np.testing.assert_array_equal(G.from_dev(d_sad2, np.uint32)[:n], want_sad[perm], err_msg=msg)
                check_winners(G.from_dev(d_best, B.ME_RESULT_DTYPE)[:nb], want_sad, want_cost, cands, offs)
                if pattern in ("max_vs_zero", "zero_vs_max") and not use_satd:
                    # the padding replicates the constant, so every candidate in range sees it
                    assert (want_sad[want_cost != EMPTY] == w * h * ((1 << bd) - 1)).all()
        free(dcur, dref)


FS_CASES = [(16, 16, 48, 16, 4), (8, 8, 20, 12, 4), (64, 64, 16, 8, 4), (16, 8, 16, 8, 4), (16, 16, 12, 4, 1)]


@pytest.mark.parametrize("bd", BDS)
def test_full_search_full_contrast(bd):
    W, H, PAD = 192, 128, 96
    c = G.ctx()
    for k, pattern in enumerate(PATTERNS):
        cur, ref, ocur, dcur, oref, dref = planes(pattern, W, H, PAD, bd, seed=30 + k)
        for w, h, rx, ry, step in FS_CASES:
            blocks = G.grid_blocks(W, H, w, h)
            want = O.full_search_blocks(ocur, oref, blocks, w, h, rx, ry, step, LAM)
            d_best = G.dev_empty(16 * len(blocks))
            c.me_full_search_dev(dcur, dref, G.to_dev(blocks), len(blocks), B.me_params(w, h, W, H, LAM, bit_depth=bd),
                                 rx, ry, step, d_best)
            c.synchronize()
            got = G.from_dev(d_best, B.ME_RESULT_DTYPE)[:len(blocks)]
            for f in ("cost", "sad", "mv_row", "mv_col"):
                np.testing.assert_array_equal(got[f], want[f], err_msg=f"{pattern} {w}x{h} {f}")
        free(dcur, dref)


SEARCH_CASES = [(16, 16, 3, 24), (8, 8, 3, 24), (32, 16, 1, 0), (4, 4, 3, 24), (16, 64, 3, 16), (64, 16, 1, 0)]


@pytest.mark.parametrize("bd", BDS)
def test_search_stages_full_contrast(bd):
    W, H, PAD = 192, 128, 160
    c = G.ctx()
    for k, pattern in enumerate(PATTERNS):
        cur, ref, ocur, dcur, oref, dref = planes(pattern, W, H, PAD, bd, seed=50 + k)
        for w, h, nsub, umh in SEARCH_CASES:
            blocks = G.grid_blocks(W, H, w, h)
            n = len(blocks)
            preds, offs = predictor_subsets(n, nsub, seed=3 + w + k, max_px=24)
            rng = np.random.default_rng(5 + k)
            pmv = (rng.integers(-40, 41, (n, 4)) * 4).astype(np.int16)
            thresh = rng.integers(0, (w * h) << (bd - 8 + 3), n).astype(np.uint32) if nsub == 3 else None
            want = O.full_pixel_me_blocks(ocur, oref, blocks, preds, offs, nsub, w, h, LAM, pmv, thresh, umh)
            d_best = G.dev_empty(16 * n)
            c.me_search_dev(dcur, dref, G.to_dev(blocks), n, G.to_dev(preds) if len(preds) else None, G.to_dev(offs),
                            nsub, B.me_params(w, h, W, H, LAM, bit_depth=bd), d_best, G.to_dev(pmv),
                            G.to_dev(thresh) if thresh is not None else None, umh)
            c.synchronize()
            got = G.from_dev(d_best, B.ME_RESULT_DTYPE)[:n]
            for f in ("cost", "sad", "mv_row", "mv_col"):
                np.testing.assert_array_equal(got[f], want[f], err_msg=f"{pattern} {w}x{h} {f}")
        free(dcur, dref)


def diamond_cands(blocks, seed):
    nb = len(blocks)
    rng = np.random.default_rng(seed)
    centre = rng.integers(-20, 21, (nb, 2)) * 8
    pattern = np.array([(0, 0)] + [(r * s, q * s) for s in (4, 2, 1) for r, q in ((1, 0), (0, 1), (-1, 0), (0, -1))])
    cands = np.zeros(nb * len(pattern), B.CAND_DTYPE)
    cands["block"] = np.repeat(np.arange(nb, dtype=np.uint32), len(pattern))
    mv = centre[:, None, :] + pattern[None, :, :]
    cands["mv_row"], cands["mv_col"] = mv[:, :, 0].reshape(-1), mv[:, :, 1].reshape(-1)
    offs = (np.arange(nb + 1) * len(pattern)).astype(np.uint32)
    pmv = (rng.integers(-64, 65, (nb, 4)) * 2).astype(np.int16)
    return cands, offs, pmv


@pytest.mark.parametrize("bd", BDS)
def test_subpel_candidates_full_contrast(bd):
    """8-tap MC of 0/max planes (the i16 intermediate at its largest) + SAD / SATD + cost."""
    W, H, PAD = 192, 128, 160
    c = G.ctx()
    for k, pattern in enumerate(PATTERNS):
        cur, ref, ocur, dcur, oref, dref = planes(pattern, W, H, PAD, bd, seed=70 + k)
        for w, h, use_satd, mode in ((16, 16, True, 0), (8, 8, False, 1), (32, 16, True, 2), (64, 64, True, 3),
                                     (8, 16, False, 0)):
            blocks = G.grid_blocks(W, H, w, h)
            nb = len(blocks)
            cands, offs, pmv = diamond_cands(blocks, seed=4 + k)
            want_sad, want_cost = O.subpel_candidates(ocur, oref, blocks, cands, w, h, use_satd, LAM, pmv,
                                                      allow_hp=True, filter_mode=mode, bit_depth=bd)
            p = B.me_params(w, h, W, H, LAM, allow_hp=True, use_satd=use_satd, bit_depth=bd)
            d_sad, d_cost, d_best = G.dev_empty(4 * len(cands)), G.dev_empty(8 * len(cands)), G.dev_empty(16 * nb)
            c.me_subpel_candidates_dev(dcur, dref, G.to_dev(blocks), nb, G.to_dev(cands), len(cands), p, mode,
                                       G.to_dev(offs), G.to_dev(pmv), d_sad, d_cost, d_best)
            c.synchronize()
            msg = f"{pattern} {w}x{h}"
            np.testing.assert_array_equal(G.from_dev(d_sad, np.uint32)[:len(cands)], want_sad, err_msg=msg)
            np.testing.assert_array_equal(G.from_dev(d_cost, np.uint64)[:len(cands)], want_cost, err_msg=msg)
            check_winners(G.from_dev(d_best, B.ME_RESULT_DTYPE)[:nb], want_sad, want_cost, cands, offs)
        free(dcur, dref)


def subpel_residual_coeffs(cur, oref, blocks, mvs, n, mode, ts, tt, bd):
    """oracle put_8tap of each block's vector -> diff -> forward_transform"""
    resid = np.zeros((len(blocks), n, n), np.int16)
    for b in range(len(blocks)):
        mr, mc = int(mvs[b][0]), int(mvs[b][1])
        x, y = int(blocks[b]["x"]), int(blocks[b]["y"])
        pred = O.put_8tap(oref, x + (mc >> 3), y + (mr >> 3), n, n, (mc << 1) & 15, (mr << 1) & 15, mode, mode, bd)
        resid[b] = cur[y:y + n, x:x + n].astype(np.int32) - pred.astype(np.int32)
    return O.forward_transform_batch(resid, ts, tt, bd, coeff_i32=(bd > 8)).reshape(len(blocks), n * n)


@pytest.mark.parametrize("bd", BDS)
def test_subpel_rdo_full_contrast(bd):
    """b200_subpel_rdo_dev (sub-pel search fused with the winner's residual and forward transform)."""
    import torch
    W, H, PAD = 192, 128, 96
    c = G.ctx()
    for k, pattern in enumerate(PATTERNS):
        cur, ref, ocur, dcur, oref, dref = planes(pattern, W, H, PAD, bd, seed=90 + k)
        for n, use_satd, tt in ((8, True, 3), (16, True, 1), (16, False, 9), (32, True, 0)):
            mode = (k + n) % 4
            ts = {8: 1, 16: 2, 32: 3}[n]
            blocks = G.grid_blocks(W, H, n, n)
            nb = len(blocks)
            cands, offs = G.random_cands(nb, 9, 6, seed=5 + k, fullpel=False)
            pmv = (np.random.default_rng(3 + k).integers(-16, 17, (nb, 4)) * 2).astype(np.int16)
            want_sad, want_cost = O.subpel_candidates(ocur, oref, blocks, cands, n, n, use_satd, LAM, pmv,
                                                      filter_mode=mode, bit_depth=bd)
            p = B.me_params(n, n, W, H, LAM, use_satd=use_satd, bit_depth=bd)
            d_sad, d_cost, d_best = G.dev_empty(4 * len(cands)), G.dev_empty(8 * len(cands)), G.dev_empty(16 * nb)
            d_coef = torch.full((nb, n * n), 77, dtype=torch.int16 if bd == 8 else torch.int32, device="cuda")
            c.subpel_rdo_dev(dcur, dref, G.to_dev(blocks), nb, G.to_dev(cands), len(cands), G.to_dev(offs), p, mode,
                             ts, tt, G.to_dev(pmv), d_sad, d_cost, d_best, d_coef)
            c.synchronize()
            msg = f"{pattern} n={n}"
            np.testing.assert_array_equal(G.from_dev(d_sad, np.uint32)[:len(cands)], want_sad, err_msg=msg)
            np.testing.assert_array_equal(G.from_dev(d_cost, np.uint64)[:len(cands)], want_cost, err_msg=msg)
            best = G.from_dev(d_best, B.ME_RESULT_DTYPE)[:nb]
            check_winners(best, want_sad, want_cost, cands, offs)
            have = best["cost"] != EMPTY
            want_coef = subpel_residual_coeffs(cur, oref, blocks, np.stack([best["mv_row"], best["mv_col"]], 1),
                                               n, mode, ts, tt, bd)
            coef = d_coef.cpu().numpy()
            np.testing.assert_array_equal(coef[have], want_coef[have], err_msg=msg)
            assert (coef[~have] == 0).all()
        free(dcur, dref)


@pytest.mark.parametrize("bd", BDS)
def test_subpel_search_full_contrast(bd):
    """b200_subpel_search_dev == the oracle's subpel_diamond_search from the same full-pel starts,
    incl. the transform of the final vector's residual."""
    import ctypes as C
    import torch
    W, H, PAD = 192, 128, 96
    c = G.ctx()
    L = O.lib()
    L.orc_subpel_diamond_search_blocks.restype = None
    L.orc_subpel_diamond_search_blocks.argtypes = [C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_ssize_t] + [C.c_int] * 3 + \
        [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_void_p] + [C.c_int] * 3 + [C.c_void_p, C.c_int]
    for k, pattern in enumerate(PATTERNS):
        cur, ref, ocur, dcur, oref, dref = planes(pattern, W, H, PAD, bd, seed=110 + k)
        for n, use_satd, allow_hp in ((16, True, True), (8, False, False)):
            ts = {8: 1, 16: 2}[n]
            blocks = G.grid_blocks(W, H, n, n)
            nb = len(blocks)
            rng = np.random.default_rng(8 + k)
            cands = np.zeros(nb, B.CAND_DTYPE)
            cands["block"] = np.arange(nb)
            cands["mv_row"], cands["mv_col"] = rng.integers(-3, 4, nb) * 8, rng.integers(-3, 4, nb) * 8
            pmv = (rng.integers(-8, 9, (nb, 4)) * 2).astype(np.int16)
            sad, cost = O.fullpel_candidates(ocur, oref, blocks, cands, n, n, False, LAM, pmv, allow_hp=allow_hp)
            start = np.zeros(nb, B.ME_RESULT_DTYPE)
            start["cost"], start["sad"], start["mv_row"], start["mv_col"] = cost, sad, cands["mv_row"], cands["mv_col"]
            want = start.copy()
            L.orc_subpel_diamond_search_blocks(ocur.origin_ptr(), ocur.stride, oref.origin_ptr(), oref.stride, ocur.bpp,
                                               2 * ((W + 7) >> 3), 2 * ((H + 7) >> 3), O.ptr(blocks), nb, n, n,
                                               int(use_satd), LAM, O.ptr(pmv), int(allow_hp), 0, bd, O.ptr(want), 0)
            p = B.me_params(n, n, W, H, LAM, allow_hp=allow_hp, use_satd=use_satd, bit_depth=bd)
            d_best = G.dev_empty(16 * nb)
            d_coef = torch.zeros((nb, n * n), dtype=torch.int16 if bd == 8 else torch.int32, device="cuda")
            c.subpel_search_dev(dcur, dref, G.to_dev(blocks), nb, G.to_dev(start), p, d_best, 0, ts, 0, G.to_dev(pmv),
                                d_coef)
            c.synchronize()
            got = G.from_dev(d_best, B.ME_RESULT_DTYPE)[:nb]
            for f in ("cost", "sad", "mv_row", "mv_col"):
                np.testing.assert_array_equal(got[f], want[f], err_msg=f"{pattern} n={n} {f}")
            want_coef = subpel_residual_coeffs(cur, oref, blocks, np.stack([want["mv_row"], want["mv_col"]], 1),
                                               n, 0, ts, 0, bd)
            np.testing.assert_array_equal(d_coef.cpu().numpy(), want_coef, err_msg=pattern)
        free(dcur, dref)


# ---------------------------------------------------------------- 2. forward transform extremes

@pytest.mark.parametrize("bd", BDS)
def test_forward_transform_extremes(bd):
    """Every valid pair on constant, checkerboard and basis-sign inputs at +-max: CUDA == oracle for
    both coefficient types at 8 bit, and the i32 output within the float model's tolerance (the i16
    one is the reference's truncating cast of it)."""
    c = G.ctx()
    for ts, tt in O.valid_txfm_combos():
        x = fwd_extreme_inputs(ts, tt, bd)
        for i32 in ([False, True] if bd == 8 else [True]):
            want = O.forward_transform_batch(x, ts, tt, bd, coeff_i32=i32)
            got = c.fwd_txfm_batch(x, ts, tt, bd, coeff_i32=i32)
            assert got.dtype == want.dtype
            np.testing.assert_array_equal(got, want, err_msg=f"ts={ts} tt={tt} i32={i32}")
            if i32 and tt != 16:
                assert_near_float_model(got, x, ts, tt, bd)


@pytest.mark.parametrize("bd", BDS)
def test_fused_residual_transform_full_contrast(bd):
    """b200_fwd_txfm_residual_dev on 0/max planes, every valid pair, zero and full-pel motion."""
    import torch
    c = G.ctx()
    W, H, PAD = 128, 128, 64
    for k, pattern in enumerate(PATTERNS):
        cur, ref, ocur, dcur, oref, dref = planes(pattern, W, H, PAD, bd, seed=130 + k)
        for ts, tt in O.valid_txfm_combos():
            w, h = O.TX_SIZES[ts]
            blocks = G.grid_blocks(W, H, w, h)
            n = len(blocks)
            rng = np.random.default_rng(ts + k)
            best = np.zeros(n, B.ME_RESULT_DTYPE)
            best["mv_col"], best["mv_row"] = rng.integers(-9, 10, n) * 8, rng.integers(-9, 10, n) * 8
            best["mv_col"][::3] = best["mv_row"][::3] = 0
            resid = np.zeros((n, h, w), np.int16)
            for i, b in enumerate(blocks):
                x, y = int(b["x"]) + PAD, int(b["y"]) + PAD
                dx, dy = int(best["mv_col"][i]) // 8, int(best["mv_row"][i]) // 8
                resid[i] = ocur.data[y:y + h, x:x + w].astype(np.int32) - oref.data[y + dy:y + dy + h, x + dx:x + dx + w]
            want = O.forward_transform_batch(resid, ts, tt, bd, coeff_i32=(bd > 8))
            d_out = torch.empty((n, w * h), dtype=torch.int32 if bd > 8 else torch.int16, device="cuda")
            c.fwd_txfm_residual_dev(dcur, dref, G.to_dev(blocks), n, G.to_dev(best), d_out, ts, tt, bd)
            c.synchronize()
            got = d_out.cpu().numpy()
            np.testing.assert_array_equal(got, want, err_msg=f"{pattern} ts={ts} tt={tt}")
            if bd > 8 and tt != 16:
                assert_near_float_model(got, resid, ts, tt, bd)
        free(dcur, dref)


# ---------------------------------------------------------------- 3. quantize chain

@pytest.mark.parametrize("ts", range(19))
def test_quantize_chain_extremes(ts):
    """qcoeffs, rcoeffs, eob and tx_dist == oracle for extreme and worst-case-spectrum coefficients,
    the three scan classes, intra and inter, 10/12-bit and mixed step sizes (the CPU suite pins the
    oracle to the typed Python model on the same inputs)."""
    for tt in SCAN_TYPES:
        for dtype, coeffs in quant_inputs(ts, tt).items():
            for dcq, acq in STEPS:
                for intra in (True, False):
                    want = oracle_chain(coeffs, ts, tt, dcq, acq, intra)
                    got = quantize_gpu(coeffs, ts, tt, dcq, acq, intra)
                    for g, w_, name in zip(got, want, ("qcoeffs", "rcoeffs", "eob", "tx_dist")):
                        np.testing.assert_array_equal(
                            g, w_, err_msg=f"{name} ts={ts} tt={tt} {dtype.__name__} {dcq}/{acq} intra={intra}")


# ---------------------------------------------------------------- 4. inverse transform at the clamps

@pytest.mark.parametrize("bd", BDS)
def test_inverse_transform_add_at_the_clamps(bd):
    """Every valid pair on coefficients across the row clamp, beyond the i32 wrap of the rectangular
    scaling and on full-scale spectra, added into planes at 0 and at max."""
    import torch
    c = G.ctx()
    px = pixel_dtype(bd)
    for ts, tt in O.valid_txfm_combos():
        w, h = O.TX_SIZES[ts]
        coef = inverse_inputs(ts, tt, bd, seed=ts * 17 + tt)
        n = len(coef)
        d_coef, d_blocks = torch.from_numpy(coef).cuda(), G.to_dev(side_by_side_blocks(n, w))
        for base_v in (0, (1 << bd) - 1):
            base = np.full((h, n * w), base_v, px)
            want = inverse_reference(coef, base, ts, tt, bd)
            dpl = c.plane_from_host(base, 0)
            c.inverse_transform_add_dev(d_coef, dpl, d_blocks, n, ts, tt, bd)
            c.synchronize()
            got = download(c, dpl, base)
            c.plane_free(dpl)
            np.testing.assert_array_equal(got, want, err_msg=f"ts={ts} tt={tt} base={base_v}")


# ---------------------------------------------------------------- 5. fused chains at 12 bit

ENC_PAIRS = [(2, 0), (1, 3), (0, 1), (3, 0), (4, 0), (9, 0), (13, 1), (5, 9), (16, 9), (11, 0), (8, 10), (14, 4),
             (3, 9), (17, 0)]


@pytest.mark.parametrize("bd", [10, 12])
@pytest.mark.parametrize("ts,tt", ENC_PAIRS)
def test_encode_tx_blocks_against_oracle_chain(ts, tt, bd):
    """b200_encode_tx_blocks_dev == the oracle's forward_transform -> quantize chain -> inverse_add into
    the prediction, every output, on full-contrast and smooth planes with 10/12-bit step sizes."""
    import torch
    c = G.ctx()
    W, H, PAD = 128, 128, 64
    w, h = O.TX_SIZES[ts]
    blocks = G.grid_blocks(W, H, w, h)
    n = len(blocks)
    rng = np.random.default_rng(ts * 7 + tt)
    mv = np.zeros(n, B.ME_RESULT_DTYPE)
    mv["cost"] = 1
    mv["mv_row"], mv["mv_col"] = rng.integers(-5, 6, n) * 8, rng.integers(-5, 6, n) * 8
    d_blocks, d_mv = G.to_dev(blocks), G.to_dev(mv)
    coded = c.L.b200_coded_tx_area(ts)
    ct = coeff_dtype(bd)
    mk = lambda k: torch.empty((n, k), dtype=torch.int32, device="cuda")
    for k, source in enumerate(PATTERNS + ["smooth"]):
        if source == "smooth":
            cur, ref = G.make_planes(W, H, PAD, pixel_dtype(bd), seed=ts, bit_depth=bd)
        else:
            cur, ref = full_scale_planes(source, W, H, bd, seed=ts + k)
        ocur, dcur = G.both_planes(cur, PAD)
        oref, dref = G.both_planes(ref, PAD)
        resid = np.zeros((n, h, w), np.int16)
        for i, b in enumerate(blocks):
            x, y = int(b["x"]) + PAD, int(b["y"]) + PAD
            dx, dy = int(mv["mv_col"][i]) // 8, int(mv["mv_row"][i]) // 8
            resid[i] = ocur.data[y:y + h, x:x + w].astype(np.int32) - oref.data[y + dy:y + dy + h, x + dx:x + dx + w]
        coef = O.forward_transform_batch(resid, ts, tt, bd, coeff_i32=True).reshape(n, w * h)
        for j, (dcq, acq) in enumerate(STEPS[1:5]):
            intra = (j + k) % 2 == 0
            wq, wr, we, wd = oracle_chain(coef, ts, tt, dcq, acq, intra)
            want_rec = ref.copy()
            for i, b in enumerate(blocks):
                x, y = int(b["x"]), int(b["y"])
                want_rec[y:y + h, x:x + w] = inverse_add(wr[i], np.ascontiguousarray(want_rec[y:y + h, x:x + w]),
                                                         ts, tt, bd)
            co, q, r = mk(w * h), mk(coded), mk(coded)
            e = torch.zeros(n, dtype=torch.int16, device="cuda")
            d = torch.zeros(n, dtype=torch.int64, device="cuda")
            rec = c.plane_from_host(ref, 0)
            c.encode_tx_blocks_dev(dcur, dref, rec, d_blocks, n, d_mv, ts, tt, bd, dcq, acq, intra, True, co, q, r, e, d)
            c.synchronize()
            msg = f"{source} {dcq}/{acq} intra={intra}"
            np.testing.assert_array_equal(co.cpu().numpy(), coef, err_msg=msg)
            np.testing.assert_array_equal(q.cpu().numpy(), wq.astype(ct), err_msg=msg)
            np.testing.assert_array_equal(r.cpu().numpy(), wr.astype(ct), err_msg=msg)
            np.testing.assert_array_equal(e.cpu().numpy().view(np.uint16), we, err_msg=msg)
            np.testing.assert_array_equal(d.cpu().numpy().view(np.uint64), wd, err_msg=msg)
            np.testing.assert_array_equal(download(c, rec, ref), want_rec, err_msg=msg)
            c.plane_free(rec)
        free(dcur, dref)


@pytest.mark.parametrize("dcq,acq", [(5347, 7312), (21387, 29247)])
def test_frame_pipe_12bit_full_contrast(dcq, acq):
    """A 12-bit b200_frame_pipe with 12-bit step sizes on full-contrast frames: push and push_packed
    against the oracle run on the same frames and lists (as test_frame_pipe_gpu does at 8 bit)."""
    W, H, PAD = 320, 176, 96
    NS, NT = 24, 6
    c = B.Context(0)
    mk = lambda: B.FramePipe(c, W, H, PAD, (16, 16), LAM, NS, NT, 40, tx_size=2, tx_type=0, dc_quant=dcq,
                             ac_quant=acq, bit_depth=12)
    dense, packed_pipe = mk(), mk()
    nb = dense.nblocks
    blocks = G.grid_blocks(W, H, 16, 16)
    assert nb == len(blocks)
    rng = np.random.default_rng(dcq)
    so = rng.integers(-40, 41, (nb, NS, 2)).astype(np.int8)
    to = rng.integers(-40, 41, (nb, NT, 2)).astype(np.int8)
    cen = (rng.integers(-6, 7, (nb, 2)) * 8).astype(np.int16)
    packed_pipe.set_lists(so, to, cen)
    scan = np.zeros(256, np.uint16)
    OL().orc_scan_order(2, 0, scan.ctypes.data, None)
    frames = [full_scale_planes(p, W, H, 12, seed=f)[f % 2]
              for f, p in enumerate(["binary", "checker", "max_vs_zero", "binary", "zero_vs_max", "checker"])]
    dense.push(frames[0])
    assert packed_pipe.push_packed(frames[0]) == 0
    for f in range(1, len(frames)):
        best, best2 = np.zeros(nb, B.ME_RESULT_DTYPE), np.zeros(nb, B.ME_RESULT_DTYPE)
        q = np.zeros((nb, 256), np.int32)
        eob, dist = np.zeros(nb, np.uint16), np.zeros(nb, np.uint64)
        dense.push(frames[f], so, to, cen, best, best2, q, eob, dist)
        g1, g2 = np.zeros(nb, B.ME_RESULT_DTYPE), np.zeros(nb, B.ME_RESULT_DTYPE)
        e2, d2 = np.zeros(nb, np.uint16), np.zeros(nb, np.uint64)
        buf = np.full(nb * 256, -1, np.int32)
        total = packed_pipe.push_packed(frames[f], g1, g2, e2, d2, buf)
        c.synchronize()
        ocur, oref = O.Plane(W, H, PAD, np.uint16), O.Plane(W, H, PAD, np.uint16)
        ocur.fill_from(frames[f])
        oref.fill_from(frames[f - 1])
        for offs, per, satd, got, got_p in ((so, NS, False, best, g1), (to, NT, True, best2, g2)):
            cands = np.zeros(nb * per, B.CAND_DTYPE)
            cands["block"] = np.repeat(np.arange(nb, dtype=np.uint32), per)
            mv = (cen[:, None, :].astype(np.int32) + 8 * offs.astype(np.int32)).astype(np.int16).reshape(-1, 2)
            cands["mv_row"], cands["mv_col"] = mv[:, 0], mv[:, 1]
            sad, cost = O.fullpel_candidates(ocur, oref, blocks, cands, 16, 16, satd, LAM)
            check_winners(got, sad, cost, cands, np.arange(nb + 1, dtype=np.uint32) * per)
            np.testing.assert_array_equal(got_p, got)
        resid = np.zeros((nb, 16, 16), np.int16)
        for i, b in enumerate(blocks):
            x, y = int(b["x"]) + PAD, int(b["y"]) + PAD
            dx, dy = int(best[i]["mv_col"]) // 8, int(best[i]["mv_row"]) // 8
            resid[i] = ocur.data[y:y + 16, x:x + 16].astype(np.int32) - oref.data[y + dy:y + dy + 16, x + dx:x + dx + 16]
        coef = O.forward_transform_batch(resid, 2, 0, 12).reshape(nb, 256)
        wq, _, we, wd = oracle_chain(coef, 2, 0, dcq, acq, False)
        np.testing.assert_array_equal(q, wq, err_msg=f"frame {f}")
        np.testing.assert_array_equal(eob, we)
        np.testing.assert_array_equal(dist, wd)
        np.testing.assert_array_equal(e2, we)
        np.testing.assert_array_equal(d2, wd)
        assert total == int(we.astype(np.int64).sum())
        np.testing.assert_array_equal(buf[:total], np.concatenate([wq[b][scan[:we[b]]] for b in range(nb)]))
        assert (buf[total:] == -1).all()
    dense.close()
    packed_pipe.close()
    c.close()
