#!/usr/bin/env python
"""bench.py — measures BASELINE.json's metric: Mpixels/s of JPEG q=80 4:2:0 encode of
3840x2160 RGB frames (config C2), per GPU and aggregated over N GPUs (one process per GPU).

A "step" is one pass of the hot path over one batch of FRAMES distinct synthetic 4K frames
(a ring larger than the 126 MB L2, so no step finds its input or output resident).

 value     device-resident throughput of the whole hot path: pixo_b200_jpeg_encode_dev =
           fused colour->subsample->DCT->quantise kernel + single-pass Huffman/stuffing
           kernel, RGB frames already in HBM -> entropy-coded scan bytes left in HBM; Mpix/s.
 e2e       the same metric through the reference-facing C ABI call with HOST buffers:
           pixo_b200_jpeg_encode_batch(pinned RGB frames) -> finished JPEG byte streams in host
           memory; H2D of the pixels, transform + Huffman/stuffing kernels, D2H of the scan bytes
           and the host-side header writing are all inside the timed region.  e2e.single_call_pageable
           is the drop-in call a pixo caller makes: pixo_b200_jpeg_encode on ONE ordinary (pageable)
           numpy frame.
 roofline  achieved HBM GB/s of the transform kernel (algorithmic 6 B/px) vs MEASURED_PEAKS, plus
           the whole device step's algorithmic bytes / time.
 cpu_baseline  the CPU restatement of pixo's encoder (oracle/, kind "port" — no Rust toolchain
           exists to build pixo itself) on the host cores, bounded sample.
 configs   the other BASELINE configurations in the same run (SURVEY.md section 8d): C3 256x1080p
           q in {50,80,95}, C4 one 16384^2 frame (band-sharded over the ranks, distributed entropy
           stage over NCCL when N > 1), C5 64x4K RGBA PNG filter + Adler-32 (frame-sharded, plus one
           image in row bands with a cross-rank Adler combine), pixo's default preset 4:4:4 q75 —
           each with Mpix/s, the kernel's roofline fraction and `bytes_identical`, a check of sample
           frames (first / middle / last of the batch) against the CPU oracle, the checker.

`--impl reference` times that CPU encoder alone (all host threads, one frame per thread).

`--dump-outputs DIR` writes what the last timed step of `value` returned (see dump_outputs), so two
builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H, QUALITY = 3840, 2160, 80
PIX = W * H
IN_BYTES = PIX * 3
ALGO_BYTES_PER_FRAME = IN_BYTES + (4 + 1 + 1) * (W // 16) * (H // 16) * 128  # 6 B/px = 49 766 400
METRIC = "Mpixels/sec JPEG q=80 4:2:0 encode of 3840x2160 RGB"


def make_frames(n: int) -> np.ndarray:
    """Ring of n distinct frames: even k = gradient shifted by k rows, odd k = LCG noise seed 42+k
    (SURVEY.md §8d generators)."""
    from pixo_b200 import synthetic
    g = synthetic.gradient_rgb(W, H).reshape(H, W * 3)
    out = np.empty((n, IN_BYTES), np.uint8)
    for k in range(n):
        if k % 2 == 0:
            out[k] = np.roll(g, k, axis=0).reshape(-1)
        else:
            out[k] = synthetic.noise(W, H, 3, 42 + k)
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        mhz, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 6:
                continue
            try:
                mhz.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(mhz)) if mhz else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(mhz)}


def measured_peak_gbs() -> tuple[float, str]:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def bind_to_gpu_numa_node(local_rank: int) -> dict:
    """Pin this rank's host threads (and therefore its first-touch pinned allocations) to the NUMA
    node its GPU hangs off: with 8 ranks each driving ~50 GB/s of H2D, buffers on the wrong socket
    cross the inter-socket link and the e2e number stops scaling (round-1 VERDICT, weak point 8)."""
    info = {"node": None, "cpus": None}
    try:
        import torch
        p = torch.cuda.get_device_properties(local_rank)
        bus = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return info
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & set(os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            info = {"node": node, "cpus": len(allowed)}
    except Exception as e:  # topology files absent (containers): stay unbound
        info["error"] = str(e)[:80]
    return info


# ------------------------------------------------------------------------------------------
def cpu_reference_rate(frames: np.ndarray, threads: int, rounds: int) -> tuple[float, float, int]:
    """The CPU encoder (oracle restatement of pixo::jpeg::encode, q80 4:2:0 baseline) on
    `threads` host threads, one whole frame per thread per round (pixo's baseline encode_scan is
    single-threaded per image, so frame-level parallelism is all the host threads it can use).
    Returns (Mpix/s, seconds, frames encoded)."""
    from oracle import pyoracle as po
    po.lib()
    n = frames.shape[0]
    bufs = [np.empty(po._jpeg_cap(W, H) // 16, np.uint8) for _ in range(threads)]
    done = [0] * threads

    def work(t):
        for r in range(rounds):
            k = (t + r * threads) % n
            cap = bufs[t].size
            ln = po.lib().po_jpeg_encode(frames[k].ctypes.data_as(po.u8p), IN_BYTES, W, H, po.RGB, QUALITY,
                                         po.S420, 0, 0, bufs[t].ctypes.data_as(po.u8p), cap)
            assert ln > 0, ln
            done[t] += 1

    ths = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
    t0 = time.perf_counter()
    for th in ths: th.start()
    for th in ths: th.join()
    dt = time.perf_counter() - t0
    nf = sum(done)
    return nf * PIX / dt / 1e6, dt, nf


def host_threads() -> int:
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0)) or n
    except AttributeError:
        pass
    return n


def best_thread_count(frames: np.ndarray) -> tuple[int, dict]:
    """The CPU arm gets the thread count it runs fastest with: all hardware threads, or one per
    physical core when SMT siblings only fight over the FP units (one calibration round each)."""
    n = host_threads()
    tried = {}
    for t in sorted({n, max(1, n // 2)}, reverse=True):
        tried[t] = cpu_reference_rate(frames, t, 1)[0]
    return max(tried, key=tried.get), tried


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    frames = make_frames(min(16, max(2, host_threads())))
    threads, tried = best_thread_count(frames)   # doubles as the warm-up
    t_total, f_total = 0.0, 0
    for _ in range(args.steps):
        _, dt, nf = cpu_reference_rate(frames, threads, 1)
        t_total += dt; f_total += nf
    rate = f_total * PIX / t_total / 1e6
    sample = (f"{threads} frames of 3840x2160 per step (one per thread), {args.steps} steps; thread count chosen "
              f"by calibration {({k: round(v) for k, v in tried.items()})} Mpix/s")
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": "Mpix/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_total / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "C2: 3840x2160 RGB -> JPEG q=80 4:2:0 baseline, standard Huffman "
                               "(frames: gradient shifted / LCG noise alternating)",
                   "frames_per_step": threads, "note": "CPU restatement of pixo's encoder "
                   "(oracle/pixo_oracle.c, gcc -O2 strict binary32); pixo itself cannot be built here (no Rust)"},
        "cpu_baseline": {"value": rate, "unit": "Mpix/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------
class Env:
    """What every measurement needs: rank/world, device, context on a torch stream, timing helpers."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.affinity0 = os.sched_getaffinity(0)
        self.numa = bind_to_gpu_numa_node(self.local_rank)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        import pixo_b200
        from pixo_b200 import _lib
        self._lib = _lib
        self.lib = _lib.load()
        self.ctx = pixo_b200.Context(self.local_rank)
        self.stream = torch.cuda.Stream(device=self.dev)
        torch.cuda.set_stream(self.stream)
        self.ctx.set_stream(self.stream.cuda_stream)
        self.peak, self.peak_src = measured_peak_gbs()

    def check(self, rc):
        self._lib.check(self.ctx.handle, rc)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def reduce_max(self, vals):
        t = self.torch.tensor(vals, dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def all_true(self, ok: bool) -> bool:
        t = self.torch.tensor([1 if ok else 0], dtype=self.torch.int64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return bool(int(t[0]))

    def timed(self, fn, steps: int, warm: int = 3) -> float:
        """ms per step, CUDA events on the launching stream, barrier + synchronize on both sides,
        max over ranks."""
        for _ in range(warm):
            fn()
        e0 = self.torch.cuda.Event(enable_timing=True)
        e1 = self.torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record(self.stream)
        for _ in range(steps):
            fn()
        e1.record(self.stream)
        self.barrier()
        return self.reduce_max([e0.elapsed_time(e1)])[0] / steps


DUMP_SAMPLE_BYTES = 15 << 20   # 60 MiB as float32: the whole dump stays under 64 MB
DUMP_SEED = 2160


def dump_sample_positions(total: int) -> np.ndarray:
    """Sorted positions into the concatenation of every frame's scan bytes: all of them when they fit
    DUMP_SAMPLE_BYTES, else one position drawn with DUMP_SEED from each of DUMP_SAMPLE_BYTES equal strata
    (so the sample depends on `total` alone)."""
    n = DUMP_SAMPLE_BYTES
    if total <= n:
        return np.arange(total, dtype=np.int64)
    lo = np.arange(n + 1, dtype=np.int64) * total // n
    return lo[:-1] + (np.random.default_rng(DUMP_SEED).random(n) * (lo[1:] - lo[:-1])).astype(np.int64)


def dump_outputs(out_dir: str, torch, d_scan, d_len, d_ovf) -> None:
    """What pixo_b200_jpeg_encode_dev hands its caller, as float .npy files: scan_lengths and
    scan_overflow (one value per frame) and scan_bytes_sample, the bytes at dump_sample_positions of the
    frames' scan bytes laid end to end in frame order (one step's scans are larger than the dump may be)."""
    lens = d_len.cpu().numpy().astype(np.int64)
    pos = dump_sample_positions(int(lens.sum()))
    starts = np.cumsum(lens) - lens
    frame = np.searchsorted(np.cumsum(lens), pos, side="right")
    flat = torch.from_numpy(frame * d_scan.shape[1] + pos - starts[frame]).to(d_scan.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "scan_lengths.npy"), lens.astype(np.float64))
    np.save(os.path.join(out_dir, "scan_overflow.npy"), d_ovf.cpu().numpy().astype(np.float64))
    np.save(os.path.join(out_dir, "scan_bytes_sample.npy"), d_scan.reshape(-1)[flat].cpu().numpy().astype(np.float32))


def sha(b) -> str:
    return hashlib.sha256(bytes(b)).hexdigest()


def scan_of(jpg: bytes) -> bytes:
    """entropy-coded segment of a baseline file: after the SOS header, before EOI"""
    i = 2
    while True:
        ln = int.from_bytes(jpg[i + 2:i + 4], "big")
        if jpg[i + 1] == 0xDA:
            return jpg[i + 2 + ln:-2]
        i += 2 + ln


def jpeg_config(env: Env, name: str, w: int, h: int, n_total: int, qualities, ss: int, steps: int,
                scaling: str = "strong (the batch is sharded over the ranks)") -> dict:
    """A batch of n_total frames sharded over the ranks (strong scaling): device-resident encode per
    quality, the transform kernel alone, and sample frames' scan bytes against the oracle."""
    from oracle import pyoracle as po      # checker only
    from pixo_b200 import jpeg, synthetic
    torch, lib = env.torch, env.lib
    # contiguous blocks: the frame content alternates (gradient / noise), so a round-robin split over an
    # even number of ranks would hand one rank all the noise frames and time only that rank
    mine = list(range(env.rank * n_total // env.world, (env.rank + 1) * n_total // env.world))
    n = len(mine)
    bases = [synthetic.noise(w, h, 3, 42 + k) if k % 2 else synthetic.gradient_rgb(w, h) for k in range(4)]
    # frame k of this rank is global frame mine[k]: build with that index
    rows = h
    d_bases = [torch.from_numpy(b).to(env.dev).reshape(rows, -1) for b in bases]
    d_px = torch.empty((n, w * h * 3), dtype=torch.uint8, device=env.dev)
    for k, g in enumerate(mine):
        d_px[k] = torch.roll(d_bases[g % 4], g, 0).reshape(-1)
    host_frame = lambda g: np.roll(bases[g % 4].reshape(rows, -1), g, axis=0).reshape(-1)
    in_each = w * h * 3
    ny, nc = jpeg.block_counts(w, h, 2, ss)
    algo = in_each + (ny + 2 * nc) * 128
    scan_cap = (in_each // 2 + 65536) // 256 * 256 * 2
    d_scan = torch.empty((n, scan_cap), dtype=torch.uint8, device=env.dev)
    d_len = torch.zeros(n, dtype=torch.int64, device=env.dev)
    d_ovf = torch.zeros(n, dtype=torch.int32, device=env.dev)
    d_y = torch.empty((n, ny * 64), dtype=torch.int16, device=env.dev)
    d_cb = torch.empty((n, nc * 64), dtype=torch.int16, device=env.dev)
    d_cr = torch.empty((n, nc * 64), dtype=torch.int16, device=env.dev)
    res = {"frames": n_total, "frames_per_gpu": n, "geometry": f"{w}x{h}", "subsampling": "4:2:0" if ss else "4:4:4",
           "scaling": scaling, "input_bytes_per_gpu": n * in_each, "per_quality": {}}
    ok_all = True
    for q in qualities:
        def enc():
            env.check(lib.pixo_b200_jpeg_encode_dev(env.ctx.handle, d_px.data_ptr(), in_each, n, w, h, 2, q, ss,
                                                    d_scan.data_ptr(), scan_cap, d_len.data_ptr(), d_ovf.data_ptr()))
        ms = env.timed(enc, steps)
        _, _, lq, cq = jpeg.quant_tables(q)

        def k1():
            env.check(lib.pixo_b200_jpeg_coefficients_dev(env.ctx.handle, d_px.data_ptr(), in_each, n, w, h, 2, ss,
                                                          lq.ctypes.data_as(env._lib.f32p), cq.ctypes.data_as(env._lib.f32p),
                                                          d_y.data_ptr(), ny * 64, d_cb.data_ptr(), d_cr.data_ptr(), nc * 64, 0, None))
        kms = env.timed(k1, steps)
        lens = d_len.cpu().numpy()
        ok = int(d_ovf.sum()) == 0
        for k in sorted({0, n // 2, n - 1}):
            ref = scan_of(po.jpeg_encode(host_frame(mine[k]), w, h, 2, q, ss))
            got = d_scan[k, : int(lens[k])].cpu().numpy().tobytes()
            ok = ok and got == ref
        ok = env.all_true(ok)
        ok_all = ok_all and ok
        res["per_quality"][str(q)] = {
            "mpix_s": n_total * w * h / (ms * 1e-3) / 1e6, "ms": ms,
            "kernel_ms": kms, "kernel_gbs": n * algo / (kms * 1e-3) / 1e9,
            "kernel_frac": n * algo / (kms * 1e-3) / 1e9 / env.peak, "bytes_identical": ok}
    res["bytes_identical"] = ok_all
    res["checked"] = "scan bytes of this rank's first / middle / last frame vs the CPU oracle, every rank"
    return res


def c4_config(env: Env, steps: int) -> dict:
    """One 16 384^2 frame.  N = 1: the whole frame through the single-context device path, and the
    same frame as 8 bands with the distributed entropy stage run in one process.  N > 1: band r on
    rank r, collectives over NCCL (parallel.encode_tiled)."""
    from oracle import pyoracle as po      # checker only
    from pixo_b200 import jpeg, parallel, synthetic
    torch, lib = env.torch, env.lib
    w = h = 16384
    q = 80
    # content: gradient with three 2048-row noise stripes (one straddles a band boundary)
    def rows_of(r0, r1):
        x = np.arange(w, dtype=np.uint64)[None, :]
        y = np.arange(r0, r1, dtype=np.uint64)[:, None]
        out = np.empty((r1 - r0, w, 3), np.uint8)
        out[..., 0] = (x * 255 // w).astype(np.uint8)
        out[..., 1] = np.broadcast_to((y * 255 // h).astype(np.uint8), (r1 - r0, w))
        out[..., 2] = ((x + y) * 127 // (w + h)).astype(np.uint8)
        out = out.reshape(r1 - r0, w * 3)
        for s0 in (2040, 9000, 14336):
            a, b = max(s0, r0), min(s0 + 2048, r1)
            if a < b:
                out[a - r0:b - r0] = noise_stripe[a - s0:b - s0]
        return out
    noise_stripe = synthetic.noise(w, 2048, 3, 4242).reshape(2048, w * 3)
    _, _, lq, cq = jpeg.quant_tables(q)
    lqp, cqp = lq.ctypes.data_as(env._lib.f32p), cq.ctypes.data_as(env._lib.f32p)
    nbands = 8 if env.world == 1 else env.world
    bands = parallel.plan_bands(w, h, nbands)
    my_bands = bands if env.world == 1 else [bands[env.rank]]
    # reference bytes: the oracle encodes the whole frame on rank 0 while the GPUs are measured
    ref = {}
    full_host = None
    if env.rank == 0:
        full_host = rows_of(0, h).reshape(-1)
        th = threading.Thread(target=lambda: ref.setdefault("sha", sha(po.jpeg_encode(full_host, w, h, 2, q, 1))))
        th.start()
    d_band_px, coefs = [], []
    for b in my_bands:
        px = torch.from_numpy(rows_of(b.px_row0, b.px_row1) if full_host is None else
                              full_host.reshape(h, w * 3)[b.px_row0:b.px_row1]).to(env.dev).reshape(-1)
        d_band_px.append(px)
        coefs.append((torch.empty((b.y_blocks, 64), dtype=torch.int16, device=env.dev),
                      torch.empty((b.c_blocks, 64), dtype=torch.int16, device=env.dev),
                      torch.empty((b.c_blocks, 64), dtype=torch.int16, device=env.dev)))
    env.torch.cuda.synchronize()
    out = {}

    coders = [parallel.DeviceBandCoder(env.ctx, dy, dcb, dcr, w, b.px_row1 - b.px_row0, 2, 1, b.y_blocks, b.c_blocks)
              for b, (dy, dcb, dcr) in zip(my_bands, coefs)]
    nonempty = [b.y_blocks > 0 for b in bands]

    def tiled_once():
        # transform of every band this rank owns, then the distributed entropy stage; the timed region
        # ends with the finished scan bytes on rank 0's device (like `value`, which leaves them in HBM)
        for b, px, (dy, dcb, dcr) in zip(my_bands, d_band_px, coefs):
            bh = b.px_row1 - b.px_row0
            env.check(lib.pixo_b200_jpeg_coefficients_dev(env.ctx.handle, px.data_ptr(), px.numel(), 1, w, bh, 2, 1, lqp, cqp,
                                                          dy.data_ptr(), b.y_blocks * 64, dcb.data_ptr(), dcr.data_ptr(),
                                                          b.c_blocks * 64, 0, None))
        if env.world == 1:
            out["parts"], out["hist"] = parallel.tiled_scan_parts_local(coders, False)
        else:   # stream-ordered: predictors, bit counts and offsets never leave the devices
            out["parts"], out["hist"] = parallel.tiled_scan_parts_async(coders[0], nonempty, env.rank, env.world)

    ms_tiled = env.timed(tiled_once, max(2, steps // 2), warm=2)
    if env.rank == 0:
        out["jpg"] = parallel.assemble_tiled(out["parts"], out["hist"], w, h, 2, q, 1)
    res = {"geometry": "16384x16384", "quality": q, "bands": nbands,
           "tiled": {"mpix_s": w * h / (ms_tiled * 1e-3) / 1e6, "ms": ms_tiled,
                     "what": ("band r on rank r: transform + k_huff<RAW> + splice per GPU, stream-ordered (predictors, bit counts "
                              "and offsets stay in device memory); all-gathers of 3+2+2 words and a gather of the scan bytes to "
                              "rank 0 over NCCL; one host wait (byte counts); timed until the scan bytes are on rank 0's device" if env.world > 1 else
                              "8 bands, every stage of the distributed path, run one after the other in ONE context"),
                     "nccl_ranks": env.world}}
    tiled_sha = sha(out["jpg"]) if env.rank == 0 else None
    if env.world == 1:
        d_px = torch.cat(d_band_px)
        n_in = w * h * 3
        scan_cap = (n_in // 2 + 65536) // 256 * 256
        d_scan = torch.empty(scan_cap, dtype=torch.uint8, device=env.dev)
        d_len = torch.zeros(1, dtype=torch.int64, device=env.dev)
        d_ovf = torch.zeros(1, dtype=torch.int32, device=env.dev)

        def whole():
            env.check(lib.pixo_b200_jpeg_encode_dev(env.ctx.handle, d_px.data_ptr(), n_in, 1, w, h, 2, q, 1, d_scan.data_ptr(),
                                                    scan_cap, d_len.data_ptr(), d_ovf.data_ptr()))
        ms_whole = env.timed(whole, max(2, steps // 2), warm=2)
        ny, nc = jpeg.block_counts(w, h, 2, 1)
        dy = torch.empty(ny * 64, dtype=torch.int16, device=env.dev)
        dcb = torch.empty(nc * 64, dtype=torch.int16, device=env.dev)
        dcr = torch.empty(nc * 64, dtype=torch.int16, device=env.dev)

        def k1():
            env.check(lib.pixo_b200_jpeg_coefficients_dev(env.ctx.handle, d_px.data_ptr(), n_in, 1, w, h, 2, 1, lqp, cqp,
                                                          dy.data_ptr(), ny * 64, dcb.data_ptr(), dcr.data_ptr(), nc * 64, 0, None))
        kms = env.timed(k1, max(2, steps // 2), warm=2)
        whole_scan = d_scan[: int(d_len.cpu()[0])].cpu().numpy().tobytes()
        res["whole_frame_one_gpu"] = {"mpix_s": w * h / (ms_whole * 1e-3) / 1e6, "ms": ms_whole, "kernel_ms": kms,
                                      "kernel_frac": 6.0 * w * h / (kms * 1e-3) / 1e9 / env.peak,
                                      "scan_sha_matches_tiled": sha(whole_scan) == sha(scan_of(out["jpg"]))}
    ok = True
    if env.rank == 0:
        th.join()
        ok = tiled_sha == ref["sha"]
        res["jpeg_bytes"] = len(out["jpg"])
    res["bytes_identical"] = env.all_true(ok)
    res["checked"] = "sha256 of the complete JPEG vs the CPU oracle's encode of the whole frame (rank 0)"
    return res


def c5_config(env: Env, steps: int) -> dict:
    """64 x 4K RGBA: PNG filter selection + fused Adler-32, frames sharded over the ranks; plus ONE
    4K RGBA image cut into row bands (one per rank, the raw row above each band is its only overlap)
    with the per-band Adler-32 values combined across ranks."""
    from oracle import pyoracle as po      # checker only
    from pixo_b200 import parallel, png, synthetic
    torch, lib = env.torch, env.lib
    w, h, bpp, n_total = 3840, 2160, 4, 64
    rb = w * bpp
    # contiguous blocks: the frame content alternates (gradient / noise), so a round-robin split over an
    # even number of ranks would hand one rank all the noise frames and time only that rank
    mine = list(range(env.rank * n_total // env.world, (env.rank + 1) * n_total // env.world))
    n = len(mine)
    g3 = synthetic.gradient_rgb(w, h).reshape(h, w, 3)
    bases = [synthetic.noise(w, h, 4, 42 + k) if k % 2 else
             np.concatenate([g3, np.full((h, w, 1), 255, np.uint8)], -1).reshape(-1) for k in range(4)]
    d_bases = [torch.from_numpy(b).to(env.dev).reshape(h, rb) for b in bases]
    d_in = torch.empty((n, h * rb), dtype=torch.uint8, device=env.dev)
    for k, g in enumerate(mine):
        d_in[k] = torch.roll(d_bases[g % 4], g, 0).reshape(-1)
    host_frame = lambda g: np.roll(bases[g % 4].reshape(h, rb), g, axis=0).reshape(-1)
    out_stride = h * (rb + 1)
    d_out = torch.empty((n, out_stride), dtype=torch.uint8, device=env.dev)
    d_ad = torch.zeros(n, dtype=torch.int32, device=env.dev)
    algo = h * rb + out_stride
    res = {"frames": n_total, "frames_per_gpu": n, "geometry": "3840x2160 RGBA", "input_bytes_per_gpu": n * h * rb,
           "scaling": "strong (the batch is sharded over the ranks)", "strategies": {}}
    ok_all = True
    for name, code in (("Adaptive", po.F_ADAPTIVE), ("AdaptiveFast", po.F_ADAPTIVE_FAST)):
        def run():
            env.check(lib.pixo_b200_png_filter_dev(env.ctx.handle, d_in.data_ptr(), h * rb, n, w, h, rb, bpp, code,
                                                   d_out.data_ptr(), out_stride, d_ad.data_ptr()))
        ms = env.timed(run, steps)
        ad = d_ad.cpu().numpy().view(np.uint32)
        ok = True
        for k in sorted({0, n // 2, n - 1}):
            ref = po.apply_filters(host_frame(mine[k]), w, h, bpp, code)
            ok = ok and sha(d_out[k].cpu().numpy().tobytes()) == sha(ref.tobytes()) and int(ad[k]) == po.adler32(ref)
        ok = env.all_true(ok)
        ok_all = ok_all and ok
        res["strategies"][name] = {"mpix_s": n_total * w * h / (ms * 1e-3) / 1e6, "ms": ms,
                                   "kernel_gbs": n * algo / (ms * 1e-3) / 1e9,
                                   "kernel_frac": n * algo / (ms * 1e-3) / 1e9 / env.peak, "bytes_identical": ok}
    # one image in row bands, Adler-32 combined across ranks
    img = host_frame(1).reshape(h, rb)
    r0, r1 = h * env.rank // env.world, h * (env.rank + 1) // env.world
    d_rows = torch.from_numpy(np.ascontiguousarray(img[r0:r1])).to(env.dev)
    d_above = torch.from_numpy(np.ascontiguousarray(img[r0 - 1])).to(env.dev) if r0 else None
    d_bout = torch.empty((r1 - r0) * (rb + 1), dtype=torch.uint8, device=env.dev)
    d_bad = torch.zeros(1, dtype=torch.int32, device=env.dev)
    gathered = {}

    def band():
        png.apply_filters_rows_dev(d_rows, d_above, w, h, r1 - r0, rb, bpp, png.FilterStrategy.Adaptive, d_bout, d_bad, ctx=env.ctx)
        t = torch.stack([d_bad[0].to(torch.int64) & 0xFFFFFFFF, torch.tensor(d_bout.numel(), dtype=torch.int64, device=env.dev)])
        if env.world > 1:
            parts = [torch.empty_like(t) for _ in range(env.world)]
            env.dist.all_gather(parts, t)
        else:
            parts = [t]
        gathered["parts"] = parts
    ms_band = env.timed(band, steps)
    parts = [(int(p[0]), int(p[1])) for p in gathered["parts"]]
    ref = po.apply_filters(img.reshape(-1), w, h, bpp, po.F_ADAPTIVE)
    mine_ok = d_bout.cpu().numpy().tobytes() == ref[r0 * (rb + 1): r1 * (rb + 1)].tobytes()
    res["one_image_row_bands"] = {"bands": env.world, "mpix_s": w * h / (ms_band * 1e-3) / 1e6, "ms": ms_band,
                                  "adler_identical": parallel.adler32_combine(parts) == po.adler32(ref),
                                  "bytes_identical": env.all_true(mine_ok),
                                  "collective": "all_gather of (adler32, length) per band, combined in band order"}
    res["bytes_identical"] = ok_all and res["one_image_row_bands"]["adler_identical"] and res["one_image_row_bands"]["bytes_identical"]
    res["checked"] = "filtered stream + Adler-32 of this rank's first / middle / last image vs the CPU oracle, every rank"
    return res


def run_ours(args):
    env = Env()
    torch, dist, lib, ctx = env.torch, env.dist, env.lib, env.ctx
    rank, world, dev, stream = env.rank, env.world, env.dev, env.stream
    from pixo_b200 import jpeg
    _lib = env._lib

    F = args.frames
    frames_host = make_frames(F)
    pinned = torch.from_numpy(frames_host).pin_memory()
    d_px = pinned.to(dev, non_blocking=True)
    ny, nc = jpeg.block_counts(W, H, 2, 1)
    d_y = torch.empty((F, ny * 64), dtype=torch.int16, device=dev)
    d_cb = torch.empty((F, nc * 64), dtype=torch.int16, device=dev)
    d_cr = torch.empty((F, nc * 64), dtype=torch.int16, device=dev)
    _, _, lq, cq = jpeg.quant_tables(QUALITY)
    lqp, cqp = lq.ctypes.data_as(_lib.f32p), cq.ctypes.data_as(_lib.f32p)

    scan_cap = IN_BYTES // 2 + 65536 + 8192
    scan_cap -= scan_cap % 256
    d_scan = torch.empty((F, scan_cap), dtype=torch.uint8, device=dev)
    d_slen = torch.zeros(F, dtype=torch.int64, device=dev)
    d_sovf = torch.zeros(F, dtype=torch.int32, device=dev)

    def encode_step():
        env.check(lib.pixo_b200_jpeg_encode_dev(ctx.handle, d_px.data_ptr(), IN_BYTES, F, W, H, 2, QUALITY, 1,
                                                d_scan.data_ptr(), scan_cap, d_slen.data_ptr(), d_sovf.data_ptr()))

    def kernel_step():
        env.check(lib.pixo_b200_jpeg_coefficients_dev(ctx.handle, d_px.data_ptr(), IN_BYTES, F, W, H, 2, 1, lqp, cqp,
                                                      d_y.data_ptr(), ny * 64, d_cb.data_ptr(), d_cr.data_ptr(),
                                                      nc * 64, 0, None))   # natural order: the launch an encode step makes

    barrier = env.barrier
    sampler = ClockSampler(env.local_rank)
    if rank == 0:
        sampler.start()
    # ---- device-resident whole path (value) ----
    for _ in range(max(args.warmup, 3)):
        encode_step()
    barrier()
    assert int(d_sovf.sum()) == 0, "scan capacity overflow"
    launches_enc0 = ctx.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for _ in range(args.steps):
        encode_step()
    ev1.record(stream)
    barrier()
    enc_launches = ctx.launch_count - launches_enc0
    enc_ms = env.reduce_max([ev0.elapsed_time(ev1)])[0]
    scan_bytes = int(d_slen.sum())
    if args.dump_outputs and rank == 0:   # every rank encodes the same frames
        dump_outputs(args.dump_outputs, torch, d_scan, d_slen, d_sovf)

    # ---- the dominant kernel alone (roofline) ----
    for _ in range(3):
        kernel_step()
    barrier()
    launches0 = ctx.launch_count
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    e_all0, e_all1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e_all0.record(stream)
    for a, b in evs:
        a.record(stream); kernel_step(); b.record(stream)
    e_all1.record(stream)
    barrier()
    kernel_launches = ctx.launch_count - launches0
    total_ms = e_all0.elapsed_time(e_all1)
    per_launch_ms = float(np.mean([a.elapsed_time(b) for a, b in evs]))
    total_ms, per_launch_ms = env.reduce_max([total_ms, per_launch_ms])
    value = world * F * args.steps * PIX / (enc_ms * 1e-3) / 1e6
    k1_value = world * F * args.steps * PIX / (total_ms * 1e-3) / 1e6

    # ---- end-to-end through the C ABI with host buffers ----
    e2e_frames = min(F, args.e2e_frames)
    cap = 2 * IN_BYTES
    out_host = torch.empty((e2e_frames, cap), dtype=torch.uint8).pin_memory()
    lens = (C.c_size_t * e2e_frames)()

    def e2e_step():
        env.check(lib.pixo_b200_jpeg_encode_batch(ctx.handle, pinned.data_ptr(), IN_BYTES, e2e_frames, W, H, 2, QUALITY,
                                                  1, 0, 0, out_host.data_ptr(), cap, lens))

    for _ in range(2):
        e2e_step()
    barrier()
    launches1 = ctx.launch_count
    t0 = time.perf_counter()
    e2e_steps = max(1, args.e2e_steps)
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    e2e_launches = ctx.launch_count - launches1
    e2e_value = world * e2e_frames * e2e_steps * PIX / env.reduce_max([e2e_s])[0] / 1e6
    jpeg_bytes = int(sum(lens))

    # the drop-in call: one ordinary (pageable) numpy frame per call, result in a bytes-like buffer
    one = frames_host[1].copy()                      # plain numpy memory, never registered with CUDA
    one_out = np.empty(cap, np.uint8)
    one_len = C.c_size_t()

    def single_call():
        env.check(lib.pixo_b200_jpeg_encode(ctx.handle, one.ctypes.data, IN_BYTES, W, H, 2, QUALITY, 1, 0, 0, 0, 0,
                                            one_out.ctypes.data, cap, C.byref(one_len)))
    for _ in range(3):
        single_call()
    barrier()
    t0 = time.perf_counter()
    single_n = 20
    for _ in range(single_n):
        single_call()
    single_s = env.reduce_max([time.perf_counter() - t0])[0]
    single_value = world * single_n * PIX / single_s / 1e6
    clocks = sampler.stop() if rank == 0 else None

    # ---- the other configurations (SURVEY.md section 8d), same run ----
    configs = {}
    want = [c for c in args.configs.split(",") if c] if args.configs != "none" else []
    del d_y, d_cb, d_cr, d_scan
    torch.cuda.empty_cache()
    launches_cfg0 = ctx.launch_count
    runners = {"C3": lambda: jpeg_config(env, "C3", 1920, 1080, 256, (50, 80, 95), 1, args.cfg_steps),
               "P444": lambda: jpeg_config(env, "P444", W, H, 32 * world, (75,), 0, args.cfg_steps,
                                           "weak (32 frames per GPU; pixo's default preset 4:4:4 q75)"),
               "C4": lambda: c4_config(env, args.cfg_steps),
               "C5": lambda: c5_config(env, args.cfg_steps)}
    for cname in want:
        try:
            t0 = time.perf_counter()
            configs[cname] = runners[cname]()
            configs[cname]["wall_s"] = round(time.perf_counter() - t0, 1)
        except Exception as e:   # a failing side configuration must not take the headline line with it
            configs[cname] = {"error": f"{type(e).__name__}: {e}"[:300], "bytes_identical": False}
            if world > 1:
                raise
        torch.cuda.empty_cache()
    cfg_launches = ctx.launch_count - launches_cfg0

    # ---- CPU baseline, rank 0 at N=1 only: bounded sample ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        os.sched_setaffinity(0, env.affinity0)     # the CPU arm gets every host core back
        cores, _tried = best_thread_count(frames_host)
        rate, dt, nf = cpu_reference_rate(frames_host, cores, 1)
        cpu = {"value": rate, "unit": "Mpix/s", "cores": cores, "kind": "port",
               "sample": f"{nf} frames of 3840x2160 (one per thread), {dt:.1f} s wall; CPU restatement of "
                         "pixo::jpeg::encode (oracle/), pixo itself unbuildable here (no Rust toolchain)"}

    if rank == 0:
        peak, peak_src = env.peak, env.peak_src
        achieved = ALGO_BYTES_PER_FRAME * F / (per_launch_ms * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get("k_jpeg_420_dram_bytes_per_launch")
            except Exception:
                traffic = None
        step_ms = enc_ms / args.steps
        step_algo = F * IN_BYTES + scan_bytes      # RGB in, scan bytes out: what the device step must move
        line = {
            "metric": METRIC, "value": value, "unit": "Mpix/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": step_ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"C2: 3840x2160 RGB -> JPEG q=80 4:2:0; step = ring of {F} distinct frames per GPU "
                                   f"({F * IN_BYTES / 1e6:.0f} MB in + same out, larger than L2: no flush needed)",
                       "frames_per_step_per_gpu": F, "global_frames_per_step": world * F,
                       "frame_content": "even: gradient_rgb shifted k rows; odd: LCG noise seed 42+k",
                       "l2_policy": "inputs+outputs larger than L2", "parallelism": f"dp{world} (frames sharded, no collective on the data path)",
                       "numa_binding": env.numa},
            "roofline": {"bound": "hbm", "kernel": "k_jpeg_420", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": ALGO_BYTES_PER_FRAME * F,
                         "kernel_ms_per_launch": per_launch_ms, "kernel_only_mpix_s": k1_value,
                         "share_of_step": per_launch_ms / step_ms,
                         "entropy_kernel_ms_per_step": step_ms - per_launch_ms,
                         "whole_step": {"algorithmic_bytes": step_algo, "gbs": step_algo / (step_ms * 1e-3) / 1e9,
                                        "frac": step_algo / (step_ms * 1e-3) / 1e9 / peak,
                                        "note": "RGB in + scan bytes out over the whole device step (K1 + k_huff); the "
                                                "coefficient arrays between the two kernels are extra traffic, not algorithmic"},
                         "note": "k_jpeg_420 timed alone (pixo_b200_jpeg_coefficients_dev, the same launch an encode "
                                 "step makes) on the same ring; the rest of a step is k_huff, the single-pass "
                                 "Huffman/stuffing kernel (instruction-issue bound, not HBM bound)"},
            "e2e": {"value": e2e_value, "unit": "Mpix/s", "h2d_bytes_per_step": e2e_frames * IN_BYTES,
                    "d2h_bytes_per_step": jpeg_bytes + e2e_frames * 12,
                    "frames_per_step": e2e_frames, "steps": e2e_steps, "jpeg_bytes_last_step": jpeg_bytes,
                    "api": "pixo_b200_jpeg_encode_batch (host RGB in pinned memory -> JPEG bytes on host)",
                    "single_call_pageable": {"value": single_value, "unit": "Mpix/s", "calls": single_n,
                                             "ms_per_call": single_s / single_n * 1e3,
                                             "api": "pixo_b200_jpeg_encode, one pageable numpy 4K frame in, JPEG bytes out, per call"}},
            "gpu_launches": int(enc_launches + kernel_launches + e2e_launches + cfg_launches),
            "host_fallbacks": ctx.host_fallbacks,
            "clocks": clocks,
            "configs": configs,
        }
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=32, help="distinct 4K frames per step per GPU")
    ap.add_argument("--e2e-frames", type=int, default=32)
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--configs", default="C3,C4,C5,P444", help="comma list of side configurations, or 'none'")
    ap.add_argument("--cfg-steps", type=int, default=8)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
