"""Full-scale and 12-bit inputs for the integer hot path: the shared input builders, and the CPU
checks that pin the oracle (and, through the host emulation, the CUDA inverse-transform source) at
the ranges where the arithmetic runs out of bits.

The parity tests elsewhere draw smooth planes with small differences and small coefficients, so the
wrapping casts, clamps and packed lanes of the kernels never see their limits there.  The builders
here produce what real 8/10/12-bit content can reach: 0/max pixel patterns, transform inputs that
drive one coefficient to its largest value, coefficients at the i16 limits, at the inverse
transform's row clamp and beyond the point where the rectangular scaling product wraps in i32.
tests/test_zz_full_scale_gpu.py runs the same inputs through the CUDA kernels."""
import numpy as np
import pytest

from tests import oracle_lib as O
from tests.test_inv_txfm_emul import emul  # noqa: F401  (module-scoped fixture)
from tests.test_oracle_inv_txfm import inverse_add
from tests.test_oracle_quantize import L as OL
from tests.test_oracle_quantize import chain as oracle_chain
from tests.test_oracle_quantize import py_quantize
from tests.test_oracle_txfm import SHIFT_SUM, float_model, mat_1d, types_1d, unpack

BDS = [8, 10, 12]
PATTERNS = ["max_vs_zero", "zero_vs_max", "checker", "binary"]
# dc/ac step sizes: the smallest, 10-bit and 12-bit table entries (quantize/tables.rs dc_qlookup /
# ac_qlookup), the 12-bit maxima, and mixed pairs that put a tiny DC step next to a huge AC one
STEPS = [(4, 4), (1336, 1828), (5347, 7312), (21387, 29247), (4, 29247), (21387, 4)]
SCAN_TYPES = [0, 10, 11]          # DCT_DCT (default scan), V_DCT (row scan), H_DCT (column scan)
RECT_WRAP = (1 << 31) // 2896 + 1  # |c| from which raw * 2896 (inverse.rs rect scaling) wraps in i32


def pixel_dtype(bd):
    return np.uint8 if bd == 8 else np.uint16


def coeff_dtype(bd):
    return np.int16 if bd == 8 else np.int32


def full_scale_planes(pattern, width, height, bd, seed=0):
    """(cur, ref) images at full contrast: constant max against 0 and the reverse, a 0/max
    checkerboard against its inverse, or seeded random 0/max images."""
    maxv = (1 << bd) - 1
    if pattern == "max_vs_zero":
        cur, ref = np.full((height, width), maxv), np.zeros((height, width))
    elif pattern == "zero_vs_max":
        cur, ref = np.zeros((height, width)), np.full((height, width), maxv)
    elif pattern == "checker":
        cur = (np.indices((height, width)).sum(0) & 1) * maxv
        ref = maxv - cur
    elif pattern == "binary":
        rng = np.random.default_rng(seed)
        cur = rng.integers(0, 2, (height, width)) * maxv
        ref = rng.integers(0, 2, (height, width)) * maxv
    else:
        raise KeyError(pattern)
    dt = pixel_dtype(bd)
    return np.ascontiguousarray(cur.astype(dt)), np.ascontiguousarray(ref.astype(dt))


def fwd_extreme_inputs(ts, tt, bd):
    """(n, h, w) int16 residuals at +-max: constant, checkerboard, and for output coefficients
    (kv, kh) with kv, kh in {0, 1, n/2, n-1} the "basis-sign" block max * sign(row kv of the
    vertical basis) x sign(row kh of the horizontal one), which drives coefficient (kv, kh) to its
    largest magnitude.  FLIPADST sees its input reversed, so its sign pattern is reversed too."""
    w, h = O.TX_SIZES[ts]
    m = (1 << bd) - 1
    chk = (np.indices((h, w)).sum(0) & 1) * 2 - 1
    xs = [np.full((h, w), m), np.full((h, w), -m), chk * m, -chk * m]
    if tt != 16:                                       # WHT_WHT has no float model: patterns only
        vt, ht = types_1d(tt)
        sv = np.where(mat_1d(vt, h) >= 0, 1, -1)
        sh = np.where(mat_1d(ht, w) >= 0, 1, -1)
        if vt == "FLIPADST":
            sv = sv[:, ::-1]
        if ht == "FLIPADST":
            sh = sh[:, ::-1]
        for kv in sorted({0, 1, h // 2, h - 1}):
            for kh in sorted({0, 1, w // 2, w - 1}):
                xs.append(m * np.outer(sv[kv], sh[kh]))
    return np.ascontiguousarray(np.stack(xs).astype(np.int16))


def float_tolerance(ts, bd, want):
    """The bound test_oracle_txfm.test_against_float_orthonormal_model applies (random inputs), plus
    at 12 bit one unit per 2^12 of the largest coefficient: the networks' cosines carry 12 bits
    (forward_shared.rs cospi), so their error grows with the coefficient, and the basis-sign
    inputs reach 524160, about 100x what random inputs give (measured: up to 87 against 56)."""
    w, h = O.TX_SIZES[ts]
    tol = 12 * (1 << SHIFT_SUM[(w, h)]) / 2 + 8
    if bd == 12:
        tol += np.abs(want).max() / 4096
    return tol


def assert_near_float_model(coef_i32, x, ts, tt, bd):
    got = unpack(coef_i32.astype(np.int64), ts)
    want = float_model(x, ts, tt)
    err = np.abs(got - want).max()
    assert err <= float_tolerance(ts, bd, want), (ts, tt, bd, err)


def quant_extreme_coeffs(ts, dtype, seed):
    """(n, w*h) blocks at the coefficient type's limits: i16 at +-32767 and -32768; i32 at
    +-524160 (the largest 12-bit forward output) and +-2^22 (shifted by log_tx_scale 2: near 2^24)."""
    w, h = O.TX_SIZES[ts]
    area = w * h
    rng = np.random.default_rng(seed)
    if dtype == np.int16:
        lo, hi = -32768, 32767
        vals = np.array([hi, -hi, lo])
    else:
        lo, hi = -(1 << 22), 1 << 22
        vals = np.array([524160, -524160, hi, lo])
    blocks = [np.full(area, v) for v in vals]
    blocks.append(rng.choice(vals, area))
    dc = np.zeros(area, np.int64)
    dc[0] = lo
    blocks.append(dc)
    sparse = np.zeros(area, np.int64)
    k = rng.choice(area, max(area // 16, 2), replace=False)
    sparse[k] = rng.choice(vals, len(k))
    blocks.append(sparse)
    return np.ascontiguousarray(np.stack(blocks).astype(dtype))


def quant_spectra(ts, tt, bd):
    """Real worst-case spectra: the forward transform of fwd_extreme_inputs, in the coefficient type
    the encoder uses at that depth (i16 at 8 bit, truncated like the reference's `as` cast)."""
    t = tt if O.valid_txfm(ts, tt) else 0
    x = fwd_extreme_inputs(ts, t, bd)
    return O.forward_transform_batch(x, ts, t, bd, coeff_i32=(bd > 8)).reshape(len(x), -1)


def quant_inputs(ts, tt):
    """Every coefficient input section 3 of the suite uses, keyed by coefficient type."""
    return {np.int16: np.concatenate([quant_extreme_coeffs(ts, np.int16, ts), quant_spectra(ts, tt, 8)]),
            np.int32: np.concatenate([quant_extreme_coeffs(ts, np.int32, ts), quant_spectra(ts, tt, 12)])}


def inverse_inputs(ts, tt, bd, seed):
    """Coded-area coefficient blocks for the inverse transform's range limits:
    a few coefficients (or all of them) at (1 << (bd+7)) +- 64, across the row clamp at bd+8 bits;
    for 1:2 rectangles at HBD, a few coefficients with |c| >= RECT_WRAP, where raw * 2896 wraps;
    and realistic spectra of full-scale residuals.  At 8 bit the i16 type caps the first kind at its
    limits (the row clamp then cannot engage; the rectangular product cannot wrap)."""
    w, h = O.TX_SIZES[ts]
    n = min(w, 32) * min(h, 32)
    ct = coeff_dtype(bd)
    info = np.iinfo(ct)
    rng = np.random.default_rng(seed)
    lim = 1 << (bd + 7)
    out = []
    for i in range(6):
        c = np.zeros(n, np.int64)
        k = rng.choice(n, min(1 + i % 4, n), replace=False)
        c[k] = rng.choice([-1, 1], len(k)) * (lim + rng.integers(-64, 65, len(k)))
        out.append(c)
    out.append(rng.choice([-1, 1], n) * (lim + rng.integers(-64, 65, n)))
    if bd > 8 and abs(int(np.log2(w)) - int(np.log2(h))) == 1:
        for i in range(6):
            c = np.zeros(n, np.int64)
            k = rng.choice(n, min(1 + i % 4, n), replace=False)
            c[k] = rng.choice([-1, 1], len(k)) * rng.integers(RECT_WRAP, 1 << 22, len(k))
            out.append(c)
    out = [np.clip(c, info.min, info.max) for c in out]
    spec = O.forward_transform_batch(fwd_extreme_inputs(ts, tt, bd), ts, tt, bd, coeff_i32=(bd > 8))
    out.extend(spec.reshape(len(spec), -1)[:, :n].astype(np.int64))
    return np.ascontiguousarray(np.stack(out).astype(ct))


def inverse_reference(coef, base, ts, tt, bd):
    """oracle inverse_transform_add of block i into base[:, i*w:(i+1)*w]"""
    w, h = O.TX_SIZES[ts]
    want = base.copy()
    for i in range(len(coef)):
        want[:, i * w:(i + 1) * w] = inverse_add(coef[i], np.ascontiguousarray(want[:, i * w:(i + 1) * w]), ts, tt, bd)
    return want


def side_by_side_blocks(n, w):
    from rav1e_b200 import backend as B
    blocks = np.zeros(n, B.BLOCK_DTYPE)
    blocks["x"] = np.arange(n) * w
    return blocks


def hadamard_satd(org, ref):
    """get_satd (dist.rs:155-220) on int64 numpy: unnormalised 2-D Hadamard of the difference per
    4x4 chunk when min(w, h) == 4, else per 8x8 chunk; sum of |coefficients|; one final rounding.
    w and h must be multiples of the chunk size (no SAD fall-back at edges)."""
    h, w = org.shape
    size = 4 if min(w, h) == 4 else 8
    hm = np.array([[1]])
    while len(hm) < size:
        hm = np.block([[hm, hm], [hm, -hm]])
    d = org.astype(np.int64) - ref.astype(np.int64)
    d = d.reshape(h // size, size, w // size, size).transpose(0, 2, 1, 3)
    total = int(np.abs(hm @ d @ hm.T).sum())
    ln = size.bit_length() - 1
    return (total + (1 << ln >> 1)) >> ln


def wrap(v, bits):
    """two's-complement wrap of Python ints / int64 arrays to `bits` bits"""
    v = np.asarray(v, np.int64)
    return ((v + (1 << (bits - 1))) & ((1 << bits) - 1)) - (1 << (bits - 1))


def typed_chain_model(c, ts, tt, dcq, acq, intra):
    """quantize -> dequantize -> raw tx-domain distortion of one block with the reference's integer
    types, on top of test_oracle_quantize.py_quantize (which works on unbounded Python ints):
      * `c.abs() >= deadzone` is evaluated in T; in release builds i16::MIN.abs() is i16::MIN, so a
        -32768 coefficient never counts for the end of block (quantize/mod.rs:296);
      * qcoeffs and rcoeffs are `T::cast_from` (an `as` cast) of i32 values (:359, :389);
      * dequantize multiplies in i32 (:388), and the distortion squares in i32 before `as u64`
        (sign extension), summing modulo 2^64 (encoder.rs:1622-1631)."""
    bits = 16 if c.dtype == np.int16 else 32
    l = OL()
    w, h = O.TX_SIZES[ts]
    coded = l.orc_coded_tx_area(ts)
    lts = l.orc_get_log_tx_scale(ts)
    scan, iscan = np.zeros(coded, np.uint16), np.zeros(coded, np.uint16)
    l.orc_scan_order(ts, tt, scan.ctypes.data, iscan.ctypes.data)
    q, _ = py_quantize(c, scan, iscan, lts, dcq, acq, intra)
    q = np.array(q, np.int64)
    off_eob = acq * (88 if intra else 44) // 256
    deadzone = -(-(acq - off_eob) // (1 << lts))
    a = wrap(np.abs(c[:coded].astype(np.int64)), bits)          # abs in T
    em1 = int(iscan[a >= deadzone].max()) if (a >= deadzone).any() else 0
    eob = em1 + 1 if em1 > 0 else int(q[0] != 0)
    q[scan[max(eob, 1):]] = 0                                    # py_quantize may have run further
    q = wrap(q, bits)
    quant = np.full(coded, acq, np.int64)
    quant[0] = dcq
    r = wrap(wrap(q * quant + ((q >> 31) & ((1 << lts) - 1)), 32) >> lts, bits)
    d = np.concatenate([c[:coded].astype(np.int64) - r, c[coded:].astype(np.int64)])
    raw = int(wrap(d * d, 32).sum()) % (1 << 64)
    sb = 2 * (3 - lts)
    return q, r, eob, (raw + (1 << (sb - 1))) >> sb


# ---------------------------------------------------------------- independent models of the oracle

@pytest.mark.parametrize("bd", BDS)
def test_sad_and_satd_models_at_full_contrast(bd):
    """The oracle's get_sad / get_satd equal w*h*|d| on constant differences and the numpy Hadamard
    model on every pattern, for every block size the per-call symbols serve."""
    from rav1e_b200 import backend as B
    for pattern in PATTERNS:
        cur, ref = full_scale_planes(pattern, 128, 128, bd, seed=bd)
        for w, h in B.BLOCK_SIZES:
            a, b = np.ascontiguousarray(cur[:h, :w]), np.ascontiguousarray(ref[:h, :w])
            pa, pb = O.Plane(w, h, 0, a.dtype), O.Plane(w, h, 0, b.dtype)
            pa.fill_from(a)
            pb.fill_from(b)
            sad = O.get_sad(pa, 0, 0, pb, 0, 0, w, h)
            assert sad == int(np.abs(a.astype(np.int64) - b).sum())
            if pattern in ("max_vs_zero", "zero_vs_max"):
                assert sad == w * h * ((1 << bd) - 1)
            assert O.get_satd(pa, 0, 0, pb, 0, 0, w, h) == hadamard_satd(a, b), (pattern, w, h)


@pytest.mark.parametrize("bd", BDS)
def test_forward_oracle_at_extremes_near_float_model(bd):
    """Constant, checkerboard and basis-sign inputs at +-max through the oracle's forward transform,
    every valid pair: within the float orthonormal model's tolerance.  At 8 bit the i16 output is
    the i32 one truncated, so the model is checked on the i32 output."""
    for ts, tt in O.valid_txfm_combos():
        x = fwd_extreme_inputs(ts, tt, bd)
        c32 = O.forward_transform_batch(x, ts, tt, bd, coeff_i32=True)
        if tt != 16:
            assert_near_float_model(c32, x, ts, tt, bd)
        if bd == 8:
            np.testing.assert_array_equal(O.forward_transform_batch(x, ts, tt, bd, coeff_i32=False),
                                          c32.astype(np.int16))
    if bd == 12:
        # the 64-point DC of a full-scale 12-bit residual sits 127 below the inverse's row clamp
        dc = O.forward_transform_batch(np.full((1, 64, 64), 4095, np.int16), 4, 0, 12)[0, 0]
        assert dc == 524160 == (1 << 19) - 128


@pytest.mark.parametrize("ts", range(19))
def test_quantize_oracle_against_typed_model(ts):
    """The oracle's chain == typed_chain_model (py_quantize with the reference's integer types) on
    extreme and worst-case-spectrum coefficients, every scan class, intra and inter, all step sizes."""
    for tt in SCAN_TYPES:
        for dtype, coeffs in quant_inputs(ts, tt).items():
            coeffs = coeffs[::2] if len(coeffs) > 12 else coeffs
            for dcq, acq in STEPS:
                for intra in (True, False):
                    q, r, eob, dist = oracle_chain(coeffs, ts, tt, dcq, acq, intra)
                    for i, c in enumerate(coeffs):
                        wq, wr, weob, wd = typed_chain_model(c, ts, tt, dcq, acq, intra)
                        ctx = (ts, tt, dtype.__name__, dcq, acq, intra, i)
                        assert int(eob[i]) == weob, ctx
                        np.testing.assert_array_equal(q[i], wq, err_msg=str(ctx))
                        np.testing.assert_array_equal(r[i], wr, err_msg=str(ctx))
                        assert int(dist[i]) == wd, ctx


def test_typed_model_reaches_the_wrapping_cases():
    """The inputs above really exercise what typed_chain_model adds to py_quantize: an i16 -32768
    that does not count for the end of block, an rcoeff that wraps in i16, and an i32 square that
    wraps (the uncoded half of a 64-point block at 2^22)."""
    c = np.full(16, -32768, np.int16)
    _, _, eob, _ = typed_chain_model(c, 0, 0, 4, 4, True)
    assert eob == 1
    c = np.full(16, 32767, np.int16)
    _, r, _, _ = typed_chain_model(c, 0, 0, 1336, 1828, True)
    assert (r[1:] < 0).all()                      # 18 * 1828 = 32904 -> -32632
    c = np.full(64 * 64, 1 << 22, np.int32)
    _, _, _, d = typed_chain_model(c, 4, 0, 4, 4, True)
    assert d < 1 << 40                             # (2^22)^2 wraps to 0 in i32


# ---------------------------------------------------------------- inverse transform at 12 bit and at the clamps

@pytest.mark.parametrize("bd", BDS)
def test_inverse_emulation_at_the_clamps(emul, bd):  # noqa: F811
    """tests/cpp/inv_txfm_emul.cu (the CUDA inverse source replayed on the host) == the oracle for
    every valid pair on inverse_inputs, into base planes at 0 and at max (the pixel clip engages at
    both ends)."""
    px = pixel_dtype(bd)
    for ts, tt in O.valid_txfm_combos():
        w, h = O.TX_SIZES[ts]
        coef = inverse_inputs(ts, tt, bd, seed=ts * 17 + tt)
        n = len(coef)
        blocks = side_by_side_blocks(n, w)
        for base_v in (0, (1 << bd) - 1):
            base = np.full((h, n * w), base_v, px)
            want = inverse_reference(coef, base, ts, tt, bd)
            got = base.copy()
            assert emul.emul_inverse_transform_add(coef.ctypes.data, got.ctypes.data, n * w, got.itemsize,
                                                   blocks.ctypes.data, n, ts, tt, bd) == 0
            np.testing.assert_array_equal(got, want, err_msg=f"ts={ts} tt={tt} bd={bd} base={base_v}")


def test_inverse_oracle_12bit_equals_10bit_inside_the_ranges():
    """The inverse depends on the bit depth only through the row clamp (bd+8 bits), the column clamp
    (max(bd+6, 16) bits) and the pixel clip.  For coefficients of residuals within +-200 none of them
    engages at 10 or 12 bit, so the 12-bit reconstruction of a flat 2048 block, minus 2048, equals the
    10-bit one of a flat 512 block, minus 512, for every valid pair."""
    rng = np.random.default_rng(12)
    for ts, tt in O.valid_txfm_combos():
        w, h = O.TX_SIZES[ts]
        n = min(w, 32) * min(h, 32)
        res = rng.integers(-200, 201, (3, h, w)).astype(np.int16)
        coef = O.forward_transform_batch(res, ts, tt, 10, coeff_i32=True).reshape(3, -1)[:, :n]
        for c in np.ascontiguousarray(coef):
            r12 = inverse_add(c, np.full((h, w), 2048, np.uint16), ts, tt, 12).astype(np.int32) - 2048
            r10 = inverse_add(c, np.full((h, w), 512, np.uint16), ts, tt, 10).astype(np.int32) - 512
            assert np.abs(r10).max() < 500                 # no clip at 10 bit
            np.testing.assert_array_equal(r12, r10, err_msg=f"ts={ts} tt={tt}")
