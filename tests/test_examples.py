"""examples/stream_frames.cpp is the C-ABI-only walk through the frame pipe (create, resident lists, one packed push
per frame).  Here: it compiles and links against the shared library with nothing but the public header, with no
CUDA device visible it fails loudly instead of computing anything on the CPU, and on a GPU it streams frames."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "rav1e_b200")


def build(tmp_path):
    exe = str(tmp_path / "stream_frames")
    subprocess.check_call(["/usr/bin/g++", "-std=c++17", "-O1", "-Wall", os.path.join(ROOT, "examples/stream_frames.cpp"),
                           "-o", exe, "-L" + PKG, "-lb200rdo", "-Wl,-rpath," + PKG])
    return exe


def test_example_builds_and_refuses_to_run_without_a_gpu(tmp_path):
    exe = build(tmp_path)
    # an empty CUDA_VISIBLE_DEVICES hides the devices of a GPU machine as well
    r = subprocess.run([exe, "2"], capture_output=True, text=True, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode != 0 and "no CPU fallback" in r.stderr


@pytest.mark.gpu
def test_example_streams_frames_on_the_gpu(tmp_path):
    exe = build(tmp_path)
    r = subprocess.run([exe, "3"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.startswith("3 frames in "), r.stdout
