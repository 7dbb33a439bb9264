#!/usr/bin/env python
"""Time per CTU of one gang as a function of how many CTAs (SMs) are busy: n gangs of h x w pictures for n in a list.
A kernel bound by SM-local resources shows a flat curve; one that leans on a shared resource (L2 for data, spills or
instruction fetch) slows down as SMs are added.  usage: python tools/occupancy_scan.py variant h w q n1 n2 ..."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "hevc-image-encoder-lite_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import hevce_b200 as H  # noqa: E402
import simutil as S  # noqa: E402
import workloads as WL  # noqa: E402

v, h, w, q = sys.argv[1], int(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4])
gang, cluster = S.variant_gang(v)
K = WL.kodak_landscape()
H.set_variant(v)
pool = [WL.config3_image(i, K)[(37 * i) % (512 - h + 1):, (53 * i) % (768 - w + 1):][:h, :w].copy() for i in range(148 * gang // cluster)]
nctu = ((h + 31) // 32) * ((w + 31) // 32)
for ng in [int(x) for x in sys.argv[5:]]:
    imgs = pool[: ng * gang // cluster]
    ses = H.Session(0, [i.shape for i in imgs], q)
    ses.upload(imgs)
    ms = min(ses.encode() for _ in range(3))
    print(f"{v}: {ng:4d} CTAs x {gang} pictures {h}x{w} q{q}: kernel {ms:8.2f} ms, {ms / nctu:.3f} ms per CTU per gang", flush=True)
    ses.close()
