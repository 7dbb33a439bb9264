#!/usr/bin/env python
"""bench.py -- Mpixel/s encoded (bit-exact bitstream) on the BASELINE.json workloads, 1..8 B200, beside the reference's CPU build.

    python bench.py --gpus N --steps K --warmup W                       # our arm (N>1: launched by torch.distributed.run)
    python bench.py --impl reference --gpus N --steps K --warmup W      # the reference's own CPU implementation
    python bench.py --config 3 --total 8192 [--gpus N]                  # configs[2] as written: 8192 pictures, strong scaling
    python bench.py --config 4 --qpd6 0|4                               # configs[3]: 64 pictures 3840x2160 (split over ranks)
    python bench.py --config 5 --mode crop|xl                           # configs[4]: one 15991x11993 picture (one GPU)
    python bench.py ... --dump-outputs DIR                              # also write the last timed step's outputs as .npy

A "step" is one pass of the hot path over one batch.  Default: `--images` (1036 = 148 SMs x 7 pictures per CTA) synthetic
768x512 pictures PER GPU at qpd6=2 -- a shard of BASELINE.json configs[2] (weak scaling: per-GPU work fixed; pictures are
independent, no collective on the data path, NCCL only carries the timing barrier / max-reduce).
  value : whole-job Mpixel/s with the inputs already resident in HBM (session upload outside the timed region)
  e2e   : the same metric through the public C entry point HEVCImageEncoderBatch with HOST buffers (H2D of the
          pictures, D2H of streams + reconstructions inside the timed region)
Parity gate of every run: each picture of the timed batch that has an entry in the committed manifests of the UNMODIFIED
reference (tests/golden/config{3,4,5}_manifest.json) is compared by SHA-256 of stream AND reconstruction -- in the first
warm-up step and the last timed step of the device-resident arm and in EVERY step of the end-to-end arm; all other
pictures must be identical between those steps and arms.  The number of pictures checked each way is reported.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "hevc-image-encoder-lite_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

W_INT_OPS_PER_PIXEL = 9782          # SURVEY.md section 8d: minimal (partial-butterfly) transform arithmetic, exact
KODAK_PIXELS = 768 * 512
GOLD = os.path.join(ROOT, "tests", "golden")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


def measured_traffic():
    """DRAM bytes per padded pixel of the decision kernel from the committed ncu capture (profiles/r2_traffic.json)."""
    p = os.path.join(ROOT, "profiles", "r2_traffic.json")
    return json.load(open(p)) if os.path.exists(p) else None


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], threading.Event()
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(int(float(r[0])) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[2 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(float(self.rows[0][1])), "reasons": reasons, "samples": len(sm)}


def cpu_checker():
    import refutil as R
    if os.path.exists(R.REF_SO):
        return R.ref(), "reference"
    return R.oracle(), "port"


def cpu_sample_run(imgs, q, threads):
    """Encode `imgs` with the CPU checker on `threads` host threads (ctypes releases the GIL; the reference is
    re-entrant, README.md:25-28). Returns seconds."""
    import refutil as R
    lib, _ = cpu_checker()
    t0 = time.perf_counter()
    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(lambda im: R.encode_with(lib, im, q), imgs))
    return time.perf_counter() - t0


def run_reference(a, rank, world):
    import workloads as WL
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    _, kind = cpu_checker()
    imgs = WL.config3_batch(0, cores)
    times = []
    for s in range(a.warmup + a.steps):
        dt = cpu_sample_run(imgs, a.qpd6, cores)
        if s >= a.warmup:
            times.append(dt)
    t = sum(times)
    mpx = len(imgs) * KODAK_PIXELS * len(times) / t / 1e6
    line = {
        "impl": "reference", "metric": "Mpixel/s encoded, bit-exact bitstream, Kodak-size batch", "value": mpx, "unit": "Mpixel/s",
        "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * t / len(times), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": "configs[2]: synthetic 768x512 8-bit grayscale (Kodak-derived), qpd6=2", "qpd6": a.qpd6},
        "cpu_baseline": {"value": mpx, "unit": "Mpixel/s", "cores": cores, "kind": kind,
                         "sample": f"{len(imgs)} pictures of the workload per step, one picture per host thread"},
        "e2e": {"value": mpx, "unit": "Mpixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---- workloads ------------------------------------------------------------------------------------------------------
def load_manifest(name):
    p = os.path.join(GOLD, name + "_manifest.json")
    return json.load(open(p))["pictures"] if os.path.exists(p) else {}


def make_workload(a, rank, world):
    """Returns (imgs, qpd6, golden entries per picture or None, description, scaling, max_dim)."""
    import workloads as WL
    K = WL.kodak_landscape()
    if a.config == 3:
        if a.total:
            lo, hi = WL.shard_range(a.total, rank, world)
            scaling, what = "strong", f"configs[2]: {a.total} synthetic 768x512 pictures split over {world} GPU(s)"
        else:
            lo, hi = rank * a.images, (rank + 1) * a.images
            scaling, what = "weak", "configs[2] shard: synthetic 768x512 8-bit grayscale (Kodak-derived, tests/workloads.py)"
        man = load_manifest("config3") if a.qpd6 == 2 else {}
        imgs = [WL.config3_image(i, K) for i in range(lo, hi)]
        gold = [man.get(f"{i:04d}") for i in range(lo, hi)]
        return imgs, a.qpd6, gold, what + f", qpd6={a.qpd6}", scaling, 8192
    if a.config == 4:
        lo, hi = WL.shard_range(a.total or 64, rank, world)
        man = load_manifest("config4")
        imgs = [WL.config4_image(i, K) for i in range(lo, hi)]
        gold = [man.get(str(i), {}).get(f"q{a.qpd6}") for i in range(lo, hi)]
        return imgs, a.qpd6, gold, f"configs[3]: {a.total or 64} synthetic 3840x2160 pictures (padded to 3840x2176), qpd6={a.qpd6}", "strong", 8192
    man = load_manifest("config5")
    imgs = [WL.config5_image(K)] if rank == 0 else []
    xl = a.mode == "xl"
    what = ("configs[4]: one synthetic 15991x11993 picture, qpd6=2, " +
            ("size limit raised to 16384: padded to 16000x12000" if xl else "drop-in limit: the top-left 8192x8192 is encoded (HEVCe.c:1581-1582)"))
    return imgs, 2, [man.get("xl" if xl else "crop")] * len(imgs), what, "strong", 16384 if xl else 8192


def sha(b):
    return hashlib.sha256(b).hexdigest()


def digests(streams, rcons):
    return [(len(s), sha(bytes(s)), sha(r.tobytes())) for s, r in zip(streams, rcons)]


def gate(dg, gold, base, where):
    """dg: digests of one step; gold: manifest entries (or None) per picture; base: digests every step must repeat."""
    n_gold = 0
    for i, (d, g) in enumerate(zip(dg, gold)):
        if g is not None:
            n_gold += 1
            if d != (g["len"], g["stream_sha256"], g["rcon_sha256"]):
                raise SystemExit(f"bench.py: PARITY FAILURE ({where}): picture {i} differs from the reference manifest")
        if base is not None and d != base[i]:
            raise SystemExit(f"bench.py: PARITY FAILURE ({where}): picture {i} differs between steps / arms")
    return n_gold


DUMP_RCON_BYTES, DUMP_STREAM_BYTES = 40 << 20, 20 << 20     # float32 payload; with the lengths the dump stays under 64 MB


def dump_outputs(d, streams, rcons):
    """--dump-outputs: what the caller of the timed path received from its last step, so that two builds can be compared
    output for output.  stream_len.npy (float64) holds every picture's stream length.  For a sample of pictures drawn with
    a fixed seed from the picture count and sizes alone (the same pictures whatever the build computes), rcon_NNNN.npy
    holds the reconstruction and stream_NNNN.npy the stream bytes, both float32.  An array larger than its share of the
    budget is written as every k-th element of its flattened form, k the smallest step that fits."""
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "stream_len.npy"), np.array([len(s) for s in streams], np.float64))
    picks, px = [], 0
    for i in np.random.default_rng(0).permutation(len(rcons)):
        if picks and px + rcons[i].size > DUMP_RCON_BYTES // 4:
            break
        picks.append(int(i))
        px += rcons[i].size
    for i in picks:
        for kind, a, room in (("rcon", rcons[i], DUMP_RCON_BYTES // 4),
                              ("stream", np.frombuffer(bytes(streams[i]), np.uint8), DUMP_STREAM_BYTES // 4 // len(picks))):
            k = max(1, -(-a.size // room))
            np.save(os.path.join(d, f"{kind}_{i:04d}.npy"), (a if k == 1 else a.reshape(-1)[::k]).astype(np.float32))


def run_one_call(a, H, WL, torch):
    """One process, one HEVCImageEncoderBatch call, N devices (hevce_api.c shards by CTU count, two chunk workers per device)."""
    nd = a.one_call
    if torch.cuda.device_count() < nd:
        raise SystemExit(f"bench.py: --one-call {nd} needs {nd} visible GPUs")
    H.set_devices(list(range(nd)))
    K = WL.kodak_landscape()
    n = a.images * nd
    imgs = [WL.config3_image(i, K) for i in range(n)]
    man = load_manifest("config3") if a.qpd6 == 2 else {}
    gold = [man.get(f"{i:04d}") for i in range(n)]
    shapes = [i.shape for i in imgs]
    host_out = H.alloc_outputs(shapes)
    s2, r2 = H.HEVCImageEncoderBatch(imgs, a.qpd6, outputs=host_out, copy_streams=False)      # warm-up
    base = digests(s2, r2)
    n_gold = gate(base, gold, None, "one-call arm, warm-up")
    for _ in range(max(a.warmup - 1, 0)):
        H.HEVCImageEncoderBatch(imgs, a.qpd6, outputs=host_out, copy_streams=False)
    t = 0.0
    with ClockSampler(0) as clk:
        for _ in range(a.steps):
            for d in range(nd):
                torch.cuda.synchronize(d)
            t0 = time.perf_counter()
            s2, r2 = H.HEVCImageEncoderBatch(imgs, a.qpd6, outputs=host_out, copy_streams=False)
            t += time.perf_counter() - t0
            gate(digests(s2, r2), gold, base, "one-call arm")
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, s2, r2)
    px = n * KODAK_PIXELS
    v = px * a.steps / t / 1e6
    line = {
        "metric": "Mpixel/s encoded, bit-exact bitstream, Kodak-size batch", "value": v, "unit": "Mpixel/s", "n_gpus": nd, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * t / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int32", "data": "synthetic",
        "config": {"workload": f"configs[2]: {n} synthetic 768x512 pictures, qpd6={a.qpd6}, ONE process and ONE HEVCImageEncoderBatch call over {nd} devices",
                   "pictures": n, "parallelism": f"library-internal: {nd} shards by CTU count, two chunk workers per device, no collective"},
        "e2e": {"value": v, "unit": "Mpixel/s", "h2d_bytes_per_step": sum(i.size for i in imgs),
                "d2h_bytes_per_step": sum(r.size for r in r2) + sum(len(x) for x in s2) + 8 * n,
                "api": "HEVCImageEncoderBatch (host buffers); `value` is this same end-to-end figure"},
        "gpu_launches": None, "clocks": clk.summary(),
        "parity": {"pictures": n, "checked_against_reference_manifest": n_gold, "checked_identical_across_steps": n},
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 3; --single-pass times exactly one)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=[3, 4, 5])
    ap.add_argument("--images", type=int, default=1036, help="config 3: pictures per GPU per step (1036 = 148 SMs x 7 pictures per CTA: one full wave)")
    ap.add_argument("--total", type=int, default=0, help="config 3 / 4: pictures per step over ALL GPUs (strong scaling)")
    ap.add_argument("--mode", default="crop", choices=["crop", "xl"], help="config 5: drop-in 8192 limit or raised limit")
    ap.add_argument("--qpd6", type=int, default=2)
    ap.add_argument("--cpu-sample", type=int, default=-1, help="pictures for the cpu_baseline leg (-1 = one per host core)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the streams and reconstructions of the last one as DIR/<name>.npy "
                         "(float32 / float64, under 64 MB: a fixed sample of the pictures; with several ranks, DIR/rank<r>/ each)")
    ap.add_argument("--one-call", type=int, default=0, metavar="N",
                    help="the library's own multi-GPU path: ONE process, ONE HEVCImageEncoderBatch call over N devices with N x --images "
                         "pictures (config 3); reports the end-to-end figure only (value = e2e)")
    ap.add_argument("--single-pass", action="store_true",
                    help="long single steps (configs 4-5): ONE upload + encode + download through the session calls that "
                         "HEVCImageEncoderBatch makes; value = the encode part, e2e = the whole pass, no warm-up")
    a = ap.parse_args()
    if a.single_pass and a.steps not in (None, 1):
        raise SystemExit("bench.py: --single-pass times exactly one step; drop --steps or pass --steps 1")
    if a.dump_outputs and a.impl == "reference":
        raise SystemExit("bench.py: --dump-outputs needs the GPU arms (the reference arm's batch is one picture per host core)")
    a.steps = 3 if a.steps is None else a.steps
    if a.impl == "ours" and not a.single_pass:
        a.warmup = max(a.warmup, 3)
    if a.single_pass:
        a.warmup, a.steps = 0, 1

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference":
        run_reference(a, rank, world)
        return

    import torch
    import hevce_b200 as H
    import workloads as WL
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the encoder has no CPU path")
    if a.one_call:
        return run_one_call(a, H, WL, torch)
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if not dist:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(v):
        if not dist:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    H.set_devices([local])
    imgs, q, gold, what, scaling, max_dim = make_workload(a, rank, world)
    H.set_max_dim(max_dim)
    n = len(imgs)
    shapes = [i.shape for i in imgs]
    pixels_rank = sum(H.padded(h) * H.padded(w) for h, w in shapes)      # padded luma pixels this rank encodes per step
    pixels_step = int(sum_over_ranks(float(pixels_rank)))

    # ---- device-resident arm: `value`
    kernel_ms, commit_ms = [0.0], [0.0]
    variant, grid, launches, base, n_gold = "-", 0, 0, None, 0
    clk_summary = None
    t_up = t_down = 0.0
    if n:
        t0 = time.perf_counter()
        ses = H.Session(local, shapes, q)
        variant, grid = ses.variant, ses.grid
        ses.upload(imgs)
        t_up = time.perf_counter() - t0                # configure + host staging + H2D
        for w in range(a.warmup):
            ses.encode()
            if w == 0:                                     # the first warm-up step is gated too
                base = digests(*ses.download())
                n_gold = gate(base, gold, None, "device-resident arm, first warm-up step")
        launches0 = ses.launches
        kernel_ms, commit_ms = [], []
    barrier()
    with ClockSampler(local) as clk:
        t0 = time.perf_counter()
        for _ in range(a.steps if n else 0):
            kernel_ms.append(ses.encode())             # CUDA events on the launching stream, inside the library
            commit_ms.append(ses.commit_ms)
        barrier()
        dt = time.perf_counter() - t0
    dt = max_over_ranks(dt)
    clk_summary = clk.summary()
    if n:
        launches = ses.launches - launches0
        t0 = time.perf_counter()
        out_last = ses.download()
        t_down = time.perf_counter() - t0              # D2H + host copies into caller-shaped buffers
        last = digests(*out_last)
        n_gold = gate(last, gold, base, "device-resident arm, last timed step")
        base = base or last
        if a.dump_outputs:
            dump_outputs(a.dump_outputs if world == 1 else os.path.join(a.dump_outputs, f"rank{rank}"), *out_last)
        ses.close()
    value = pixels_step * a.steps / dt / 1e6

    # ---- end-to-end arm through the public C entry point with host buffers (every step gated)
    e2e_t = 0.0
    if a.single_pass:
        e2e_t = max_over_ranks(t_up + dt + t_down)
        s2, r2 = out_last if n else ([], [])
    if n and not a.single_pass:
        host_out = H.alloc_outputs(shapes)                 # caller-owned pbuffer / img_rcon arrays, reused like a C caller would
        s2, r2 = H.HEVCImageEncoderBatch(imgs, q, outputs=host_out, copy_streams=False)   # warm-up: pooled sessions, pinned staging, page faults
        gate(digests(s2, r2), gold, base, "end-to-end arm, warm-up")
    for _ in range(0 if a.single_pass else a.steps):
        barrier()
        t0 = time.perf_counter()
        if n:
            s2, r2 = H.HEVCImageEncoderBatch(imgs, q, outputs=host_out, copy_streams=False)
        barrier()
        e2e_t += max_over_ranks(time.perf_counter() - t0)
        if n:
            gate(digests(s2, r2), gold, base, "end-to-end arm")
    e2e_value = pixels_step * a.steps / e2e_t / 1e6
    h2d = sum(i.size for i in imgs) if max_dim >= 16384 or a.config != 5 else sum(min(i.shape[0], 8192) * i.shape[1] for i in imgs)
    d2h = (sum(r.size for r in r2) + sum(len(s) for s in s2) + 8 * n) if n else 0
    stream_bytes = sum(len(s) for s in s2) if n else 0

    # ---- roofline of the decision kernel: integer issue, SURVEY.md section 8d
    km = sum(kernel_ms) / max(len(kernel_ms), 1) * 1e-3
    int_peak = H.measure_int_peak(local)
    achieved = pixels_rank * W_INT_OPS_PER_PIXEL / km if km else 0.0
    pk, pk_src = peaks()
    hbm_bytes = 2 * pixels_rank + stream_bytes           # 1 B/px read + 1 B/px recon written + bitstream
    tr = measured_traffic()
    roofline = {
        "bound": "int_issue", "kernel": f"hevce_encode_kernel_{variant}",
        "achieved": achieved / 1e12, "peak": int_peak / 1e12, "unit": "Tint-op/s", "frac": achieved / int_peak,
        "peak_source": "measured live: hevce_int_peak_kernel (IMAD=2 ops + LOP3 + IADD3 chains); MEASURED_PEAKS.json has no integer figure",
        "work_per_pixel": W_INT_OPS_PER_PIXEL, "kernel_ms": km * 1e3, "commit_kernel_ms": sum(commit_ms) / max(len(commit_ms), 1),
        "traffic": int(tr["dram_bytes_per_pixel"] * pixels_rank) if tr else None,
        "traffic_source": (f"{tr['dram_bytes_per_pixel']:.0f} B per padded pixel (dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full "
                           f"capture, {tr['source']}) x the pixels of this launch") if tr else None,
        "hbm": {"algorithmic_bytes": hbm_bytes, "achieved_gbs": hbm_bytes / km / 1e9 if km else 0.0, "peak_gbs": pk["hbm_gbs"],
                "frac": hbm_bytes / km / 1e9 / pk["hbm_gbs"] if km else 0.0, "peak_source": pk_src},
    }

    line = {
        "metric": "Mpixel/s encoded, bit-exact bitstream, Kodak-size batch" if a.config == 3 else "Mpixel/s encoded, bit-exact bitstream",
        "value": value, "unit": "Mpixel/s",
        "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * dt / a.steps, "higher_is_better": True,
        "scaling": scaling, "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": what, "pictures_this_rank": n, "qpd6": q, "pixels_per_step": pixels_step, "kernel_variant": variant, "grid_ctas": grid,
                   "l2": f"inputs larger than L2: {pixels_rank / 1e6:.0f} MB of pictures + {pixels_rank * 2.4 / 1e6:.0f} MB of per-CTU records/levels written and re-read per step",
                   "parallelism": f"{world} x independent shards, no collective"},
        "e2e": {"value": e2e_value, "unit": "Mpixel/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "api": ("one pass of hevce_session_create/upload/encode/download with host buffers -- the calls HEVCImageEncoderBatch makes; "
                        "the encode part of the same pass is `value`") if a.single_pass else
                       "HEVCImageEncoderBatch (host buffers, pinned staging inside the library)", "steps": a.steps},
        "gpu_launches": int(sum_over_ranks(float(launches))),
        "clocks": clk_summary,
        "roofline": roofline,
        "parity": {"pictures_this_rank": n, "checked_against_reference_manifest": n_gold,
                   "checked_identical_across_steps_and_arms": n, "what": "SHA-256 of stream and reconstruction, every picture; "
                   "device-resident arm: first warm-up and last timed step, end-to-end arm: every step"},
    }

    if rank == 0 and not a.no_cpu:
        cores = os.cpu_count() or 1
        _, kind = cpu_checker()
        if a.config == 3:
            m = cores if a.cpu_sample < 0 else a.cpu_sample
            sample = imgs[:m] if m <= n else WL.config3_batch(0, m)
            t = cpu_sample_run(sample, q, cores)
            line["cpu_baseline"] = {"value": len(sample) * KODAK_PIXELS / t / 1e6, "unit": "Mpixel/s", "cores": cores, "kind": kind,
                                    "sample": f"first {len(sample)} pictures of the timed batch, one per host thread, {t:.1f} s"}
        else:   # hours of CPU: the reference's time was recorded when the manifest was made (build container, one core per picture)
            secs = [g["cpu_seconds"] for g in gold if g]
            if secs:
                px = [H.padded(h) * H.padded(w) for (h, w), g in zip(shapes, gold) if g]
                line["cpu_baseline"] = {"value": sum(px) / sum(secs) / 1e6, "unit": "Mpixel/s", "cores": 1, "kind": "reference",
                                        "sample": f"{len(secs)} picture(s) of this workload, oracle/_ref on one core each in the build container "
                                                  f"while the manifest was made ({sum(secs):.0f} CPU-seconds; tests/golden manifests)"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if dist:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
