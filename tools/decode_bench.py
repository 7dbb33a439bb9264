"""Times the decoder (hevce_parse_kernel, hevce_recon_kernel, hevce_deblock_kernel) with CUDA events, and
HEVCImageDecoderBatch end to end, beside the encode time of the same batch.

Workloads: the benchmark's 1036 pictures of 768x512 at qpd6 2 (tests/workloads.py config 3) and 24 pictures of
3840x2160 at qpd6 2 (config 4).  Per workload: one encode (HEVCImageEncoderBatchDecoded, host clock), a check that the
decoder returns the encoder's decoded pictures, a warm-up, then the median of --runs kernel runs of a Decoder and of
--runs end-to-end calls.  Writes a JSON report with the card's name and power limit.

    python tools/decode_bench.py --out profiles/f6_decode_bench.json [--runs 10]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "hevc-image-encoder-lite_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import hevce_b200 as H  # noqa: E402
import workloads as WL  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:   # the report says what could not be read
        return {"error": str(e)}


def bench(name, imgs, q, runs):
    t0 = time.perf_counter()
    streams, _, decs = H.HEVCImageEncoderBatchDecoded(imgs, q)
    encode_s = time.perf_counter() - t0
    got = H.HEVCImageDecoderBatch(streams)
    assert all(np.array_equal(g, d) for g, d in zip(got, decs)), f"{name}: decoded pictures differ from the encoder's"
    pixels = sum(d.size for d in decs)
    dec = H.Decoder(0)
    dec.upload(streams)
    dec.run()                                       # warm-up
    parse, recon, dbk = [], [], []
    for _ in range(runs):
        dec.run()
        parse.append(dec.parse_ms)
        recon.append(dec.recon_ms)
        dbk.append(dec.deblock_ms)
    dec.close()
    e2e = []
    H.HEVCImageDecoderBatch(streams)                # warm-up of the cached decoder
    for _ in range(runs):
        t0 = time.perf_counter()
        H.HEVCImageDecoderBatch(streams)
        e2e.append(time.perf_counter() - t0)
    med = lambda v: float(np.median(v))
    kernels_ms = med(parse) + med(recon) + med(dbk)
    r = {
        "workload": name, "pictures": len(imgs), "qpd6": q, "padded_pixels": pixels,
        "stream_bytes": sum(len(s) for s in streams),
        "parse_ms": med(parse), "recon_ms": med(recon), "deblock_ms": med(dbk), "kernels_ms": kernels_ms,
        "kernels_mpix_per_s": pixels / kernels_ms / 1e3,
        "end_to_end_ms": med(e2e) * 1e3, "end_to_end_mpix_per_s": pixels / med(e2e) / 1e6,
        "encode_s_one_call": encode_s, "encode_mpix_per_s_one_call": pixels / encode_s / 1e6,
        "runs": runs, "spread_parse_ms": [min(parse), max(parse)], "spread_recon_ms": [min(recon), max(recon)],
    }
    print(json.dumps(r), flush=True)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--runs", type=int, default=10)
    a = ap.parse_args()
    H.set_devices([0])
    K = WL.kodak_landscape()
    rep = {"card": card(), "method": "CUDA events around each kernel of hevce_decoder_run, median of --runs after one warm-up; "
           "end to end: host clock around HEVCImageDecoderBatch (upload, kernels, download); encode: host clock around one "
           "HEVCImageEncoderBatchDecoded call of the same pictures",
           "results": [bench("config3_1036x768x512_q2", WL.config3_batch(0, 1036), 2, a.runs),
                       bench("config4_24x3840x2160_q2", [WL.config4_image(i, K) for i in range(24)], 2, a.runs)]}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rep, f, indent=1)


if __name__ == "__main__":
    main()
