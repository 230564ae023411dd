"""Y4M reader (the input format of the path, src/bin/decoder/y4m.rs): header / frame parsing on synthetic
streams of every layout, and BASELINE config 0's tests/small_input.y4m against the committed luma fixture."""
import os

import numpy as np
import pytest

from rav1e_b200 import y4m

HERE = os.path.dirname(os.path.abspath(__file__))


def make_stream(w, h, cs, nframes, seed=0):
    bd, xdec, ydec, chroma = y4m._CS[cs]
    rng = np.random.default_rng(seed)
    out = bytearray(f"YUV4MPEG2 W{w} H{h} F30:1 Ip A1:1 C{cs}\n".encode())
    want = []
    for _ in range(nframes):
        out += b"FRAME\n"
        planes = []
        sizes = [(h, w)] + ([((h + ydec) >> ydec, (w + xdec) >> xdec)] * 2 if chroma else [])
        for ph, pw in sizes:
            p = rng.integers(0, 1 << bd, (ph, pw)).astype(np.uint8 if bd == 8 else "<u2")
            out += p.tobytes()
            planes.append(p)
        want.append(planes)
    return bytes(out), want


@pytest.mark.parametrize("cs", ["420jpeg", "420p10", "422", "444p12", "mono"])
def test_roundtrip_of_synthetic_streams(cs):
    data, want = make_stream(36, 22, cs, 3, seed=len(cs))
    got = list(y4m.frames(data))
    assert len(got) == 3
    for (hdr, planes), w in zip(got, want):
        assert (hdr["width"], hdr["height"], hdr["bit_depth"]) == (36, 22, y4m._CS[cs][0])
        assert len(planes) == len(w)
        for a, b in zip(planes, w):
            np.testing.assert_array_equal(a, b)


def test_bad_streams_are_rejected():
    with pytest.raises(y4m.Y4MError):
        list(y4m.frames(b"RIFF....\n"))
    data, _ = make_stream(16, 16, "420jpeg", 1)
    with pytest.raises(y4m.Y4MError):
        list(y4m.frames(data[:-5]))
    with pytest.raises(y4m.Y4MError):
        y4m.parse_header(b"YUV4MPEG2 W16 H16 Cbogus")


def test_config0_input_matches_the_committed_fixture():
    """tests/small_input.y4m (64x64 4:2:0 8-bit, 5 frames; stored as tests/golden/small_input.y4m) -> the luma
    planes of tests/golden/small_input_luma.npy"""
    src = os.path.join(HERE, "golden", "small_input.y4m")
    luma = np.load(os.path.join(HERE, "golden", "small_input_luma.npy"))
    got = list(y4m.frames(src))
    assert len(got) == len(luma) == 5
    for (hdr, planes), want in zip(got, luma):
        assert (hdr["width"], hdr["height"], hdr["bit_depth"], hdr["xdec"], hdr["ydec"]) == (64, 64, 8, 1, 1)
        np.testing.assert_array_equal(planes[0], want)
        assert planes[1].shape == planes[2].shape == (32, 32)
