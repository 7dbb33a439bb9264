"""File-level parity of the drop-in CLI (SURVEY.md section 8f, f1): hevc-image-encoder-lite_b200/HEVCe against the
reference CLI built from the unmodified sources (oracle/_ref/HEVCe): identical .h265, identical reconstruction PGM,
identical report on stdout, same argument conventions (lone '0'..'4' anywhere = qpd6, default 3)."""
import os
import subprocess

import numpy as np
import pytest

import golden_util as G
import refutil as R

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OURS = os.path.join(ROOT, "hevc-image-encoder-lite_b200", "HEVCe")
REF = os.path.join(ROOT, "oracle", "_ref", "HEVCe")


def write_pgm(path, img):
    with open(path, "wb") as f:
        f.write(b"P5\n%d %d\n255\n" % (img.shape[1], img.shape[0]))
        f.write(np.ascontiguousarray(img, np.uint8).tobytes())


@pytest.mark.parametrize("case,args", [("k01_45x70", ["2"]), ("k01_64x128", []), ("noise_64", ["0"])])
def test_cli_matches_reference_cli(tmp_path, case, args):
    """Against the reference's stream and reconstruction in the goldens and the report figures they give; and, where
    oracle/_ref holds the reference CLI, against its .h265, reconstruction PGM and report byte for byte."""
    if not os.path.exists(OURS):
        pytest.skip("CLI binaries not built")
    data, _ = G.small_cases()
    src = tmp_path / "in.pgm"
    write_pgm(src, data[f"{case}/in"])
    outs = {}
    for tag, exe in (("ref", REF), ("ours", OURS)):
        if not os.path.exists(exe):
            continue
        h265, rec = tmp_path / f"{tag}.h265", tmp_path / f"{tag}.pgm"
        # qpd6 deliberately placed between the file names: "any lone character 0..4 is qpd6" (HEVCeMain.c:150-161)
        r = subprocess.run([exe, str(src)] + args + [str(h265), str(rec)], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stdout + r.stderr
        report = r.stdout.replace(str(h265), "<stream>").replace(str(rec), "<rcon>")
        outs[tag] = (h265.read_bytes(), rec.read_bytes(), report)
    if "ref" in outs:
        assert outs["ours"][0] == outs["ref"][0]
        assert outs["ours"][1] == outs["ref"][1]
        assert outs["ours"][2] == outs["ref"][2]
    q = int(args[0]) if args else 3
    want_s, want_r = data[f"{case}/q{q}/stream"].tobytes(), data[f"{case}/q{q}/rcon"]
    assert outs["ours"][0] == want_s
    assert np.array_equal(R.read_pgm(str(tmp_path / "ours.pgm")), want_r)
    report = outs["ours"][2].splitlines()
    assert f"  Qp%6                            = {q}     (Qp={6 * q + 4})" in report
    for line in R.report_figures(data[f"{case}/in"], want_r, len(want_s)):
        assert line in report, line
