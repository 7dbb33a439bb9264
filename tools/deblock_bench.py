#!/usr/bin/env python
"""Device time of the in-loop deblocking filter (hevce_session_deblock, hevce_deblock_kernel) beside the decision kernel
of the same batch.  Batches: the default bench workload (1,036 synthetic 768x512 pictures, qpd6 2) and 3840x2160
pictures (config 4).  Each batch is encoded once; the filter is launched `--warmup` times, then `--reps` times, each
launch timed by CUDA events.  Both batches' planes are larger than the 126 MB L2, so every launch reads from HBM.

Bytes the kernel must move: 1 B/pixel read + 1 B/pixel written, plus the CtuRec bytes it reads per CTU (its own
64 CU-size + 16 kind bytes, and one unit row, 8 + 4 bytes, of the CTUs above and below).  The halo rows and columns
a CTA reads again are not counted.
usage: python tools/deblock_bench.py [--reps 20] [--warmup 3] [--n4k 24] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "hevc-image-encoder-lite_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import hevce_b200 as H  # noqa: E402
import workloads as WL  # noqa: E402

REC_BYTES_PER_CTU = 64 + 16 + 2 * (8 + 4)


def device_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True)
    if out.returncode != 0:
        raise SystemExit(f"nvidia-smi failed: {out.stderr.strip()}")
    name, power, clock = (v.strip() for v in out.stdout.strip().split(","))
    return {"device": name, "power_limit": power, "max_sm_clock": clock}


def measure(name, imgs, q, reps, warmup):
    ses = H.Session(0, [i.shape for i in imgs], q)
    ses.upload(imgs)
    kernel_ms = ses.encode()
    commit_ms = ses.commit_ms
    for _ in range(warmup):
        ses.deblock()
    ms = np.array([ses.deblock() for _ in range(reps)])
    ses.close()
    px = sum(H.padded(i.shape[0]) * H.padded(i.shape[1]) for i in imgs)
    nbytes = 2 * px + REC_BYTES_PER_CTU * px // 1024
    med = float(np.median(ms))
    return {
        "batch": name, "pictures": len(imgs), "qpd6": q, "padded_pixels": px, "bytes": nbytes, "launches": reps,
        "deblock_ms_median": med, "deblock_ms_min": float(ms.min()), "deblock_ms_max": float(ms.max()),
        "mpixel_per_s": px / med / 1e3, "gb_per_s": nbytes / med / 1e6,
        "decision_kernel_ms": kernel_ms, "commit_kernel_ms": commit_ms,
        "deblock_share_of_encode": med / (kernel_ms + commit_ms),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--n4k", type=int, default=24, help="3840x2160 pictures in the second batch")
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    a = ap.parse_args()
    if a.reps < 20:
        raise SystemExit("--reps must be at least 20")
    info = device_info()
    K = WL.kodak_landscape()
    rows = [measure("bench: 1036 x 768x512", [WL.config3_image(i, K) for i in range(1036)], 2, a.reps, a.warmup),
            measure(f"{a.n4k} x 3840x2160", [WL.config4_image(i, K) for i in range(a.n4k)], 2, a.reps, a.warmup)]
    res = {**info, "results": rows}
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
