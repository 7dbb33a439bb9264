"""The decoder's entry points in the built library without a GPU: the header check is host code and answers, decoding
has no CPU path and fails with HEVCE_ERR_CUDA."""
import os
import subprocess

import numpy as np
import pytest

import golden_util as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROG = r"""
import sys
sys.path.insert(0, sys.argv[1])
import numpy as np
import hevce_b200 as H
s = bytes.fromhex(sys.argv[2])
print(H.stream_info(s))
try:
    H.HEVCImageDecoderBatch([s])
    print("decoded")
except H.HevceError as e:
    print("error", e.code)
"""


def test_without_a_device():
    lib = os.path.join(ROOT, "hevc-image-encoder-lite_b200", "libhevce_b200.so")
    if not os.path.exists(lib):
        pytest.skip("library not built")
    npz, _ = G.small_cases()
    s = npz["k01_64x128/q3/stream"].tobytes()
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")   # no device, whatever the machine has
    r = subprocess.run(["python", "-c", PROG, os.path.join(ROOT, "hevc-image-encoder-lite_b200"), s.hex()], capture_output=True,
                       text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stderr
    out = r.stdout.split("\n")
    assert out[0] == "(64, 128, 3)"
    assert out[1] == "error -2"
