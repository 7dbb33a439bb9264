#!/usr/bin/env python
"""SSIM on the device and the quality-target entry point, measured on one GPU (DESIGN.md section 3.7).

  1. Kernel time of hevce_session_ssim (hevce_ssim_kernel + hevce_ssim_mean_kernel, one pair of CUDA events) on the
     reconstructions of the bench batch (1,036 synthetic 768x512 pictures, qpd6 2) and of 3840x2160 pictures (config 4):
     each batch is encoded once, SSIM is launched `--warmup` times, then `--reps` times; the median is reported.  Both
     batches' planes are larger than the 126 MB L2, so every launch reads from HBM.  Bytes: each CTA loads 38x38 samples
     of both planes for its 32x32 window centres (2 B/pixel plus the halo); the partials and means are not counted.
  2. For the bench batch at SSIM targets 0.90 and 0.97: the wall time of one HEVCImageEncoderBatchTarget call beside one
     HEVCImageEncoderBatch call at qpd6 2, alternated in the same run (median of `--calls` each, after one warm-up call
     of each), the probes per picture and the histogram of chosen qpd6.  The probes come from the session's decoded SSIM
     of every picture at all five qpd6 and the search rule; the chosen qpd6 must agree with it.
usage: python tools/target_bench.py [--reps 20] [--warmup 3] [--calls 3] [--n4k 24] [--out FILE]"""
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

TILE = 38 * 38   # samples of each plane one CTA loads for 32x32 window centres


def device_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True)
    if out.returncode != 0:
        raise SystemExit(f"nvidia-smi failed: {out.stderr.strip()}")
    name, power, clock = (v.strip() for v in out.stdout.strip().split(","))
    return {"device": name, "power_limit": power, "max_sm_clock": clock}


def kernel(name, imgs, q, reps, warmup):
    ses = H.Session(0, [i.shape for i in imgs], q)
    ses.upload(imgs)
    kernel_ms = ses.encode()
    for _ in range(warmup):
        ses.ssim()
    ms = []
    for _ in range(reps):
        ses.ssim()
        ms.append(ses.ssim_ms)
    ses.close()
    ms = np.array(ms)
    px = sum(H.padded(i.shape[0]) * H.padded(i.shape[1]) for i in imgs)
    nbytes = 2 * TILE * (px // 1024)
    med = float(np.median(ms))
    return {
        "batch": name, "pictures": len(imgs), "qpd6": q, "padded_pixels": px, "bytes": nbytes, "launches": reps,
        "ssim_ms_median": med, "ssim_ms_min": float(ms.min()), "ssim_ms_max": float(ms.max()),
        "mpixel_per_s": px / med / 1e3, "gb_per_s": nbytes / med / 1e6,
        "decision_kernel_ms": kernel_ms,
    }


def rule(row, target):
    lo, hi, probes = -1, 5, 0
    while hi - lo > 1:
        q = (lo + hi) // 2
        probes += 1
        if row[q] >= target:
            lo = q
        else:
            hi = q
    return (lo if lo >= 0 else 0), probes


def target_calls(imgs, targets, calls):
    rows = []
    for q in range(5):   # decoded SSIM of every picture at every qpd6
        ses = H.Session(0, [i.shape for i in imgs], q)
        ses.upload(imgs)
        ses.encode()
        ses.deblock()
        rows.append(ses.ssim(decoded=True))
        ses.close()
    rows = np.stack(rows, axis=1)
    H.HEVCImageEncoderBatch(imgs, 2)                 # warm-up: sessions, staging, first launches
    out = []
    for t in targets:
        H.HEVCImageEncoderBatchTarget(imgs, t, "ssim")
        batch_s, target_s = [], []
        for _ in range(calls):
            t0 = time.perf_counter()
            H.HEVCImageEncoderBatch(imgs, 2)
            batch_s.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            _, _, qpd6, quality = H.HEVCImageEncoderBatchTarget(imgs, t, "ssim")
            target_s.append(time.perf_counter() - t0)
        want = [rule(r, t) for r in rows]
        probes = np.array([p for _, p in want])
        out.append({
            "target_ssim": t, "pictures": len(imgs), "calls": calls,
            "target_call_s_median": float(np.median(target_s)), "batch_call_qpd6_2_s_median": float(np.median(batch_s)),
            "target_over_batch": float(np.median(target_s) / np.median(batch_s)),
            "probes_per_picture_mean": float(probes.mean()), "probes_histogram": {str(k): int((probes == k).sum()) for k in (1, 2, 3)},
            "chosen_qpd6_histogram": {str(k): int((np.asarray(qpd6) == k).sum()) for k in range(5)},
            "target_missed": int((quality < t).sum()),
            "chosen_matches_rule": bool(all(int(q) == c for q, (c, _) in zip(qpd6, want))),
        })
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--calls", type=int, default=3, help="timed calls of each entry point per target")
    ap.add_argument("--n4k", type=int, default=24, help="3840x2160 pictures in the second batch")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "f7_target_bench.json"))
    a = ap.parse_args()
    if a.reps < 20:
        raise SystemExit("--reps must be at least 20")
    info = device_info()
    H.set_devices([0])
    K = WL.kodak_landscape()
    bench = [WL.config3_image(i, K) for i in range(1036)]
    res = {**info,
           "ssim_kernel": [kernel("bench: 1036 x 768x512", bench, 2, a.reps, a.warmup),
                           kernel(f"{a.n4k} x 3840x2160", [WL.config4_image(i, K) for i in range(a.n4k)], 2, a.reps, a.warmup)],
           "target_calls": target_calls(bench, [0.90, 0.97], a.calls)}
    txt = json.dumps(res, indent=1)
    print(txt)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(txt + "\n")


if __name__ == "__main__":
    main()
