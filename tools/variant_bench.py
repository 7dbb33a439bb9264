#!/usr/bin/env python
"""Per-variant latency of the decision kernel on a full grid: 148 x gang pictures of h x w (default 64x64 = 4 CTUs) per
variant, device-resident, CUDA-event kernel time -> ms per CTU of one gang (what the variant choice in
hevce_variants.h:HEVCE_VARIANT_LIST is calibrated with).  usage: python tools/variant_bench.py [h] [w] [qpd6] [variants...]"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "hevc-image-encoder-lite_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import hevce_b200 as H  # noqa: E402
import simutil as S  # noqa: E402
import workloads as WL  # noqa: E402

h, w, q = (int(v) for v in (sys.argv[1:4] + ["64", "64", "2"][len(sys.argv[1:4]):]))
variants = sys.argv[4:] or list(S.variants())
K = WL.kodak_landscape()
base = None
for v in variants:
    gang, cluster = S.variant_gang(v)
    n = 148 * gang // cluster
    imgs = [WL.config3_image(i, K)[(37 * i) % (512 - h + 1):, (53 * i) % (768 - w + 1):][:h, :w].copy() for i in range(n)]
    H.set_variant(v)
    ses = H.Session(0, [i.shape for i in imgs], q)
    assert ses.variant == v
    ses.upload(imgs)
    ms = [ses.encode() for _ in range(3)]
    streams, _ = ses.download()
    ses.close()
    nctu = ((h + 31) // 32) * ((w + 31) // 32)
    per = min(ms) / nctu
    base = base or per
    print(f"{v}: {n} pictures {h}x{w} q{q}: kernel {min(ms):.2f} ms, {per:.3f} ms per CTU per gang, relative {per / base:.2f}, "
          f"{n * h * w / min(ms) / 1e3:.2f} Mpx/s, bytes {sum(len(s) for s in streams)}", flush=True)
H.set_variant(None)
