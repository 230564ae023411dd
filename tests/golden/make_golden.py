#!/usr/bin/env python
"""Extracts the reference's own known-answer vectors for the hot path into
tests/golden/reference_kats.json (run by hand in the build container; needs /root/reference).

Sources (xiph/rav1e @ 564ae3b):
  src/dist.rs:418-441     get_sad_same_inner   (w, h, SAD)  on the closed-form planes of :384-413
  src/dist.rs:477-500     get_satd_same_inner  (w, h, SATD)
  src/predict.rs:1523-1566  4x4 DC / DC_TOP / DC_LEFT / DC_128 / V / H / Paeth / smooth x3
  src/predict.rs:1569-1602  27 directional angles and their expected 4x4 outputs
  src/cdef.rs:304-309     first_max_element
  src/quantize/mod.rs:186-215  test_tx_log_scale (TxSize, log_tx_scale) pairs
  src/scan_order.rs:28-947     the 42 scan tables (sha256 of each, as little-endian u16) and the
                               (TxSize, TxType) -> table map of av1_scan_orders :949-1321
  src/transform/mod.rs:519-552  log_tx_ratios (TxSize, rect_ratio_log2) pairs
  src/transform/mod.rs:555-603  roundtrips: (TxSize, TxType, tolerance) of forward -> inverse_transform_add
  src/recon_intra.rs:30-136, :258-354  the 22 has_tr_* and 22 has_bl_* availability bitmaps of
                               get_intra_edges' has_top_right / has_bottom_left (length, first 4
                               bytes and sha256 of each; the oracle and the CUDA side regenerate
                               them from their rule)
  tests/small_input.y4m   BASELINE config 0's input: the luma planes of its 5 frames (64x64, 8 bit)
                          -> tests/golden/small_input_luma.npy, and the clip itself (31 KB), byte for byte
                          -> tests/golden/small_input.y4m, so that the Y4M reader is checked without rav1e
The Rust test code is parsed textually; nothing is executed (no rustc in this image).
"""
import json
import os
import re

REF = "/root/reference/src"
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_kats.json")


def triples(text):
    return [[int(a), int(b), int(c)] for a, b, c in re.findall(r"\((\d+),\s*(\d+),\s*(\d+)\)", text)]


def main():
    dist = open(os.path.join(REF, "dist.rs")).read()
    sad_part = dist[dist.index("fn get_sad_same_inner"):dist.index("fn get_sad_same_u8")]
    satd_part = dist[dist.index("fn get_satd_same_inner"):dist.index("fn get_satd_same_u8")]
    pred = open(os.path.join(REF, "predict.rs")).read()
    t = pred[pred.index("fn pred_matches_u8"):pred.index("fn pred_max")]
    arrays = re.findall(r"\[((?:\s*\d+\s*,?)+)\s*\]", t)
    nums = [[int(x) for x in re.findall(r"\d+", a)] for a in arrays]
    lists16 = [a for a in nums if len(a) == 16]
    angles = next(a for a in nums if len(a) == 27)
    # order of appearance: V, H, Paeth, smooth, smooth_h, smooth_v, then 27 directional rows
    names = ["V_PRED", "H_PRED", "PAETH_PRED", "SMOOTH_PRED", "SMOOTH_H_PRED", "SMOOTH_V_PRED"]
    fixed = dict(zip(names, lists16[:6]))
    directional = lists16[6:6 + 27]
    assert len(directional) == 27
    consts = dict(zip(["DC_PRED", "DC_TOP", "DC_LEFT", "DC_128"],
                      [int(x) for x in re.findall(r"\[(\d+)u8; 16\]", t)]))
    cdef = open(os.path.join(REF, "cdef.rs")).read()
    c = cdef[cdef.index("fn check_max_element"):]
    fme = [{"input": [int(x) for x in re.findall(r"-?\d+", inp)], "expect": [int(i), int(v)]}
           for inp, i, v in re.findall(r"first_max_element\(&\[([^\]]+)\]\),\s*\((\d+),\s*(-?\d+)\)", c)]
    import hashlib
    import struct
    q = open(os.path.join(REF, "quantize", "mod.rs")).read()
    qt = q[q.index("fn test_tx_log_scale"):]
    qt = qt[:qt.index("];")]
    log_tx_scale = [[name, int(v)] for name, v in re.findall(r"\((TX_\w+),\s*(\d+)\)", qt)]
    sc = open(os.path.join(REF, "scan_order.rs")).read()
    tables = {}
    for m in re.finditer(r"static (\w+)\s*:\s*\[u16;\s*(\d+)\]\s*=\s*\[(.*?)\];", sc, re.S):
        vals = [int(x) for x in re.findall(r"\d+", m.group(3))]
        if len(vals) == int(m.group(2)):
            tables[m.group(1)] = {"n": len(vals), "first8": vals[:8],
                                  "sha256": hashlib.sha256(struct.pack("<%dH" % len(vals), *vals)).hexdigest()}
    blk = sc[sc.index("pub static av1_scan_orders"):]
    scan_map = {sz: re.findall(r"scan: &(\w+),", body) for sz, body in re.findall(r"// (TX_\w+)\n(.*?)\],", blk, re.S)}
    assert len(tables) == 42 and len(scan_map) == 19 and all(len(v) == 16 for v in scan_map.values())
    assert len(log_tx_scale) == 19
    tm = open(os.path.join(REF, "transform", "mod.rs")).read()
    lr = tm[tm.index("fn log_tx_ratios"):tm.index("fn roundtrips")]
    log_tx_ratios = [[n, int(v)] for n, v in re.findall(r"\(TxSize::(TX_\w+),\s*(-?\d+)\)", lr)]
    rt = tm[tm.index("fn roundtrips<T: Pixel>"):tm.index("fn roundtrips_u8")]
    rt = "\n".join(l for l in rt.splitlines() if not l.strip().startswith("//"))
    roundtrips = [[a, b, int(t)] for a, b, t in re.findall(r"\((TX_\w+),\s*(\w+),\s*(\d+)\)", rt)]
    assert len(log_tx_ratios) == 19 and len(roundtrips) == 44, (len(log_tx_ratios), len(roundtrips))
    ri = open(os.path.join(REF, "recon_intra.rs")).read()
    avail = {}
    for m in re.finditer(r"static (has_(?:tr|bl)_\d+x\d+): &\[u8\] =\s*&\[(.*?)\];", ri, re.S):
        vals = [int(x) for x in re.findall(r"\d+", m.group(2))]
        avail[m.group(1)] = {"n": len(vals), "first4": vals[:4], "sha256": hashlib.sha256(bytes(vals)).hexdigest()}
    assert len(avail) == 44, sorted(avail)
    out = {
        "source": "xiph/rav1e @ 564ae3b, extracted by tests/golden/make_golden.py",
        "intra_avail_tables": avail,
        "log_tx_ratios": log_tx_ratios, "roundtrips": roundtrips,
        "log_tx_scale": log_tx_scale, "scan_tables": tables, "scan_map": scan_map,
        "dist_pattern": {"org": "(x + y + 24) & 255", "ref": "(x - y + 8) & 255", "block_at": [32, 40],
                         "derivation": "src/dist.rs:384-413 (xpad/ypad 136 and 264; alignment terms cancel)"},
        "sad": triples(sad_part), "satd": triples(satd_part),
        "intra_4x4_edge": "edge_buf[i] = max(0, i + 32 - 128), i in 0..257 (predict.rs:1516-1517)",
        "intra_4x4_const": consts, "intra_4x4": fixed,
        "directional_angles": angles, "directional_4x4": directional,
        "first_max_element": fme,
    }
    assert len(out["sad"]) == 22 and len(out["satd"]) == 22 and len(fme) == 3
    with open(OUT, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", OUT)
    # config 0: YUV4MPEG2 W64 H64 ... C420jpeg, 5 x ("FRAME\n" + 4096 Y + 1024 U + 1024 V)
    import numpy as np
    raw = open(os.path.join(os.path.dirname(REF), "tests", "small_input.y4m"), "rb").read()
    header, rest = raw.split(b"\n", 1)
    fields = dict((t[:1].decode(), t[1:].decode()) for t in header.split()[1:])
    w, h = int(fields["W"]), int(fields["H"])
    assert (w, h) == (64, 64) and fields["C"].startswith("420")
    frames = []
    while rest:
        assert rest.startswith(b"FRAME\n")
        rest = rest[6:]
        frames.append(np.frombuffer(rest[:w * h], np.uint8).reshape(h, w).copy())
        rest = rest[w * h * 3 // 2:]
    luma = np.stack(frames)
    assert luma.shape == (5, 64, 64)
    np.save(os.path.join(os.path.dirname(OUT), "small_input_luma.npy"), luma)
    print("wrote small_input_luma.npy", luma.shape, int(luma.sum()))
    with open(os.path.join(os.path.dirname(OUT), "small_input.y4m"), "wb") as f:
        f.write(raw)
    print("wrote small_input.y4m", len(raw), "bytes")


if __name__ == "__main__":
    main()
