#!/usr/bin/env python
"""A/B builds of ONE kernel variant of libhevce_b200 with other compile-time settings, timed on the same GPU.
  python tools/ab_variants.py build t1 "TRK_C=640,LPW=4,LPW_P=18" "TRK_C=576,LPW=5,LPW_P=18"     (here, no GPU needed)
  python tools/ab_variants.py run t1 [h w q]                                                          (on the GPU box)
Each spec overrides -DHEVCE_OPT_<NAME>=<value> of the variant's flags in csrc/Makefile; the other variants are linked unchanged."""
import glob
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "hevc-image-encoder-lite_b200", "csrc")
sys.path.insert(0, os.path.join(ROOT, "tests"))
import simutil as S  # noqa: E402

OUT = os.environ.get("HEVCE_AB_DIR") or os.path.join(ROOT, "hevc-image-encoder-lite_b200", "ab")
ARCH = "-gencode arch=compute_100a,code=sm_100a"
FLAGS = f"{ARCH} -O3 -lineinfo -std=c++17 -Xcompiler -fPIC,-fvisibility=hidden"


if sys.argv[1] == "build":
    tag, specs = sys.argv[2], sys.argv[3:]
    os.makedirs(OUT, exist_ok=True)
    for f in glob.glob(os.path.join(OUT, "*.so")):
        os.remove(f)
    subprocess.run(["make", "-C", CSRC], check=True, stdout=subprocess.DEVNULL)
    others = [o for o in glob.glob(os.path.join(CSRC, "hevce_k_*.o")) if not o.endswith(f"hevce_k_{tag}.o")]
    procs = []
    for spec in ["base"] + specs:
        defs = {d.split("=")[0]: d for d in S.variant_flags(tag)}
        if spec != "base":
            for kv in spec.split(","):
                k, v = kv.split("=")
                defs[f"-DHEVCE_OPT_{k}"] = f"-DHEVCE_OPT_{k}={v}"
        name = spec.replace("=", "").replace(",", "_")
        obj, so = os.path.join(OUT, name + ".o"), os.path.join(OUT, f"libhevce_{name}.so")
        cmd = (f"nvcc {FLAGS} {' '.join(defs.values())} -DHEVCE_VARIANT={tag} -DHEVCE_NS=hevce_{tag} -c -o {obj} {CSRC}/hevce_variant.cu && "
               f"nvcc {ARCH} -shared -o {so} {obj} {' '.join(others)} {CSRC}/hevce_cuda.o {CSRC}/hevce_api.o -Xlinker --exclude-libs,ALL -lpthread && rm {obj}")
        procs.append((spec, subprocess.Popen(cmd, shell=True, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for spec, p in procs:
        out, _ = p.communicate()
        print(spec, "ok" if p.returncode == 0 else "FAILED\n" + out[-3000:])
else:
    tag = sys.argv[2]
    h, w, q = (sys.argv[3:6] + ["64", "64", "2"][len(sys.argv[3:6]):])
    code = ("import sys,os; sys.path.insert(0,'hevc-image-encoder-lite_b200'); sys.path.insert(0,'tests'); import numpy as np, hevce_b200 as H, workloads as WL;"
            "H.LIB_PATH=sys.argv[1]; tag=sys.argv[2]; h,w,q,n=map(int,sys.argv[3:7]); K=WL.kodak_landscape();"
            "imgs=[WL.config3_image(i,K)[(37*i)%(512-h+1):,(53*i)%(768-w+1):][:h,:w].copy() for i in range(n)]; H.set_variant(tag);"
            "s=H.Session(0,[i.shape for i in imgs],q); s.upload(imgs); ms=[s.encode() for _ in range(4)]; st,_=s.download();"
            "import hashlib; print(os.path.basename(sys.argv[1]), ' '.join('%.2f'%m for m in ms), hashlib.sha256(b''.join(st)).hexdigest()[:12], flush=True)")
    n = str(148 * S.variant_gang(tag)[0])   # a picture per CTA slot of 148 CTAs
    for rep in range(2):
        for so in sorted(glob.glob(os.path.join(OUT, "*.so"))):
            subprocess.run([sys.executable, "-c", code, so, tag, h, w, q, n], cwd=ROOT)
