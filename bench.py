#!/usr/bin/env python
"""bench.py — inpainted frames/s at 1080p, STTN (sttn-auto, neighbor_stride 5), BASELINE.json config 2.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload ...] [--dump-outputs DIR]

A *step* is one pass of the hot path over one chunk: 50 synthetic 1920x1080 frames + the default-bbox mask (`STTNAutoInpaint`'s
clip_gap, sttn_auto_inpaint.py:242-245); the 300-frame clip of config 2 is K = 6 steps.  Prints ONE JSON line (rank 0):
  value     frames/s with the chunk's strips already resident in HBM (device work only, CUDA events on the engine's stream), on the
            attention path whose results a caller receives (config.attention, settled by one checked pass: `settle_attention_path`)
  e2e       frames/s through the reference-facing call with HOST numpy frames: host->device copy of the strips, all kernels,
            device->host copy, composite into the host frames — what STTNAutoInpaint's chunk loop does per chunk
  roofline  the dominant kernel (transformer-block 3x3 conv 256->256, tcgen05 implicit GEMM) AS IT RUNS IN THE CHUNK: one eager pass
            of the chunk with CUDA events around every launch group (vsr_sttn_profile), algorithmic FLOPs / measured time against
            the sustained bf16 peak of MEASURED_PEAKS.json; the isolated back-to-back figure is kept beside it
  cpu_baseline  the reference's own `STTNInpaint.__call__` (baseline/_ref, kind "reference") on a bounded sample on the host cores,
            or the oracle port when the reference modules did not travel (kind "port")
`--impl reference` times only that CPU path, with all host threads, on the same config.
`--dump-outputs DIR` (sttn-auto) writes what the last timed step computed, as the frames a caller of the path receives, to DIR/*.npy
(float32, see `output_sample`): the inputs are seeded, so two builds run with the same arguments can be compared output for output.
Under torchrun (N > 1) every rank owns K chunks of its own (weak scaling, no data-path collective: chunks are independent units,
SURVEY.md §8e); timing is the max over ranks.

Everything that touches CUDA goes through `BACKEND` and every engine is built by a `make_*` factory, so that tests/test_bench_dryrun.py
can run every workload and both arms on the CPU with stand-ins (a name error or a JSON-schema regression fails in `-m "not gpu"`).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W, CHUNK = 1080, 1920, 50
FLOP_PER_FRAME = 642.8e9  # SURVEY.md §8d / BASELINE.md §3 (2*MAC of conv+matmul per output frame)
METRIC = "inpainted frames/sec at 1080p (STTN, window=5)"
WORKLOAD = "STTN sttn-auto 1080p synthetic clip, fixed subtitle bbox, neighbor_stride=5 (BASELINE config 2); step = one 50-frame chunk"
CPU_BUDGET_S = 240.0      # wall-clock target of a whole `--impl reference --steps K --warmup W` run


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured"
    return 1590.0, 1400.0, 6650.0, "fallback"


# ------------------------------------------------------------------------------------------------ CUDA / torch.distributed seam
class CudaBackend:
    """torch is the container for events, streams and torch.distributed only (the engines own their device memory)."""

    def __init__(self):
        import torch

        self.torch = torch
        self.world = 1
        self.local = 0

    def available(self):
        return self.torch.cuda.is_available()

    def setup(self, local, world):
        self.local, self.world = local, world
        self.torch.cuda.set_device(local)
        if world > 1:
            import torch.distributed as dist

            dist.init_process_group("nccl", device_id=self.torch.device("cuda", local))

    def device(self):
        return self.torch.device("cuda", self.local)

    def sync(self):
        self.torch.cuda.synchronize()

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist

            dist.barrier()

    def event(self):
        return self.torch.cuda.Event(enable_timing=True)

    def stream(self, ptr):
        return self.torch.cuda.ExternalStream(ptr, device=self.device())

    def max_over_ranks(self, values):
        t = self.torch.tensor(list(values), dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            import torch.distributed as dist

            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    def finish(self):
        if self.world > 1:
            import torch.distributed as dist

            dist.destroy_process_group()


BACKEND = None   # set in main(); the dry-run test installs a stand-in


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) < 8:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ engines (factories = test seam)
def sttn_weights():
    """(what the product's constructor gets, description): the reference checkpoint when it is staged, else seeded random-init
    tensors of the architecture from the package's own shape table."""
    p = os.path.join(ROOT, "weights", "sttn-auto", "infer_model.pth")
    if os.path.exists(p):
        return p, "reference checkpoint sttn-auto/infer_model.pth"
    from vsr_b200 import synthetic as S

    return S.random_sttn_weights(0), "seeded random-init weights of the sttn-auto architecture"


def make_sttn(device):
    from vsr_b200 import STTNInpaint

    src, desc = sttn_weights()
    return STTNInpaint(device, src), src, desc


def make_sttn_det(device):
    from vsr_b200 import STTNDetInpaint
    from vsr_b200 import synthetic as S

    p = os.path.join(ROOT, "weights", "sttn-det", "sttn.pth")
    if os.path.exists(p):
        return STTNDetInpaint(device, p), "reference checkpoint sttn-det/sttn.pth"
    return STTNDetInpaint(device, S.random_sttn_weights(1)), "seeded random-init weights of the sttn-det architecture"


def detector_dir():
    d = os.path.join(ROOT, "weights", "V5", "ch_det")
    if not os.path.exists(os.path.join(d, "inference.pdiparams")):
        raise SystemExit("this workload needs weights/V5/ch_det (tools/stage_weights.py)")
    return d


def make_detector(device):
    from vsr_b200.dbnet import TextDetector

    return TextDetector(detector_dir(), device)


def make_subtitle_detect(device):
    from vsr_b200 import SubtitleDetect

    return SubtitleDetect("", model_dir=detector_dir(), device=device)


def make_lama(device):
    from vsr_b200 import LamaInpaint

    npz = os.path.join(ROOT, "weights", "big-lama", "big-lama.npz")
    if not os.path.exists(npz):
        raise SystemExit("bench.py --workload lama needs weights/big-lama/big-lama.npz (tools/stage_weights.py --lama)")
    return LamaInpaint(device, npz), npz, "reference big-lama weights (conv kernels stored fp16)"


def propainter_dir():
    mdir = os.path.join(ROOT, "weights", "propainter")
    need = ["raft-things.pth", "recurrent_flow_completion.pth"]
    ok = all(os.path.exists(os.path.join(mdir, f)) for f in need) and any(os.path.exists(os.path.join(mdir, f)) for f in ("ProPainter.pth", "ProPainter.f16.pth"))
    if not ok:
        raise SystemExit("bench.py --workload propainter needs weights/propainter/{raft-things,recurrent_flow_completion,ProPainter}.pth (tools/stage_weights.py)")
    return mdir


def make_propainter(device):
    from vsr_b200.propainter_inpaint import PropainterInpaint

    return PropainterInpaint(device, propainter_dir())


def synthetic():
    from vsr_b200 import synthetic as S

    return S


def chunk_schedule(T, stride=5, ref=10):
    """[(neighbours, refs)] of a T-frame chunk (sttn_auto_inpaint.py:142-146, get_ref_index :107-120) — pure Python, for FLOP counts."""
    out = []
    for f in range(0, T, stride):
        nb = list(range(max(0, f - stride), min(T, f + stride + 1)))
        out.append((nb, [i for i in range(0, T, ref) if i not in nb]))
    return out


# ------------------------------------------------------------------------------------------------ CPU legs (reference / port)
def reference_available():
    from oracle import ref_import

    return ref_import.available()


class CpuReference:
    """The reference's own CPU implementation of the path: `STTNInpaint(torch.device('cpu'), model_path).__call__(frames, mask)`
    (backend/inpaint/sttn_auto_inpaint.py:28-97) from the unmodified modules (oracle/ref_import.py), or — when those did not travel —
    the oracle port of the same call (oracle/sttn_oracle.py `sttn_call`)."""

    def __init__(self, weights_src, threads=None):
        import torch

        self.torch = torch
        self.default_threads = torch.get_num_threads()      # what the unmodified reference runs with when nobody sets anything
        self.threads = threads or self.default_threads
        self.swept = None
        torch.set_num_threads(self.threads)
        self.kind = "port"
        self.model = None
        if isinstance(weights_src, str) and weights_src.endswith(".pth") and reference_available():
            try:
                from oracle import ref_import

                ref_import.install()
                from backend.inpaint.sttn_auto_inpaint import STTNInpaint as RefSTTNInpaint

                self.model = RefSTTNInpaint(torch.device("cpu"), weights_src)
                self.kind = "reference"
            except Exception as e:  # e.g. a module of the reference's environment is missing on this box
                print(f"[bench] unmodified reference not usable here ({type(e).__name__}: {e}); timing the oracle port", file=sys.stderr)
        if self.model is None:
            from oracle import sttn_oracle as O

            self.O = O
            self.w = O.load_weights(weights_src) if isinstance(weights_src, str) else {k: torch.from_numpy(v) for k, v in weights_src.items()}

    def __call__(self, frames, mask):
        with self.torch.no_grad():
            if self.model is not None:
                return self.model(frames, mask)
            return self.O.sttn_call(self.w, frames, mask)

    def fps(self, frames, mask):
        t0 = time.perf_counter()
        self(frames, mask)
        dt = time.perf_counter() - t0
        return len(frames) / dt, dt

    def pick_threads(self, frames, mask):
        """torch's CPU convolutions do not scale to every hardware thread of a 100+-thread host (128 threads: 0.2 frames/s, 16 threads:
        3 frames/s on the same box): time a 4-frame call at a few thread counts and keep the fastest, so that the baseline is the best
        the host can do.  Returns the rate of the winning setting."""
        ncpu = os.cpu_count() or 1
        cands = sorted({c for c in (8, 16, 32, 64, self.default_threads, ncpu) if 1 <= c <= ncpu})
        best, best_fps, seen = self.threads, 0.0, {}
        for c in cands:
            self.torch.set_num_threads(c)
            self.fps(frames[:2], mask)                      # warm the pools of this setting
            f, _ = self.fps(frames[:4], mask)
            seen[c] = round(f, 3)
            if f > best_fps:
                best, best_fps = c, f
        self.threads, self.swept = best, seen
        self.torch.set_num_threads(best)
        return best_fps

    def describe(self):
        what = ("unmodified reference STTNInpaint.__call__ (backend/inpaint/sttn_auto_inpaint.py:43-97)" if self.kind == "reference"
                else "oracle port of STTNInpaint.__call__ (torch CPU fp32 restatement)")
        sweep = f" (fastest of a sweep, frames/s by threads: {self.swept})" if self.swept else ""
        return f"{what}, torch {self.torch.__version__} CPU fp32, {self.threads} of {os.cpu_count()} threads{sweep}"


CPU_SAMPLE_SIZES = (6, 10, 16, 25, 50)


def cpu_sample_frames(cpu, frames, mask, per_step_s):
    """Frames per CPU step, chosen by measurement: the largest of CPU_SAMPLE_SIZES whose call fits the per-step budget.  The cost per frame
    grows with the clip (attention is quadratic in the window length, and windows reach their full 10-15 frames only from ~16 frames on),
    so a rate measured on a short clip must not be extrapolated: sizes are tried in ascending order (each try doubles as warm-up) until one
    exceeds the budget or the next is predicted to (quadratic extrapolation).  Shorter samples are FASTER per frame than a whole chunk:
    the bias favours the CPU."""
    best, t_prev, n_prev = CPU_SAMPLE_SIZES[0], None, None
    for n in CPU_SAMPLE_SIZES:
        if t_prev is not None and t_prev * (n / n_prev) ** 2 > 1.5 * per_step_s:
            break
        _, t = cpu.fps(frames[:n], mask)
        if t > per_step_s and n != CPU_SAMPLE_SIZES[0]:
            break
        best, t_prev, n_prev = n, t, n
    return best


def run_reference(args, rank, world):
    if rank != 0:
        return
    S = synthetic()
    src, wdesc = sttn_weights()
    cpu = CpuReference(src)
    frames = S.synthetic_clip(CHUNK, H, W, seed=0)
    mask = S.default_mask(H, W)
    cpu.pick_threads(frames, mask)                          # thread-count sweep, doubles as the first warm-up
    n = cpu_sample_frames(cpu, frames, mask, CPU_BUDGET_S / max(args.steps + args.warmup, 1))
    for _ in range(args.warmup):
        cpu.fps(frames[:n], mask)
    dts = []
    for _ in range(args.steps):
        dts.append(cpu.fps(frames[:n], mask)[1])
    value = n * len(dts) / float(np.sum(dts))
    sample = (f"each step = the first {n} frames of the 50-frame 1080p chunk through the {cpu.describe()}; sample sized so that "
              f"{args.steps}+{args.warmup} steps take ~{CPU_BUDGET_S:.0f} s (shorter windows than a whole chunk: favours the CPU)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean(dts)), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": f"synthetic 1080p clip (seeded, generated on host); {wdesc}",
            "config": {"workload": WORKLOAD, "frame": [H, W], "chunk": CHUNK, "neighbor_stride": 5, "ref_length": 10,
                       "strip": [720, 1080, 0, 1920], "frames_per_step": n},
            "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cpu.threads, "kind": cpu.kind, "sample": sample},
            "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def cpu_baseline_leg(src, frames, mask, n_frames):
    cpu = CpuReference(src)
    cpu.pick_threads(frames, mask)                          # thread-count sweep = warm-up (thread pools, oneDNN primitives)
    fps, dt = cpu.fps(frames[:n_frames], mask)
    return {"value": fps, "unit": "frames/s", "cores": cpu.threads, "kind": cpu.kind,
            "sample": f"the first {n_frames} frames of the 50-frame 1080p chunk through the {cpu.describe()}: {dt:.1f} s of CPU work "
                      "(shorter windows than a whole chunk: favours the CPU)"}


# ------------------------------------------------------------------------------------------------ secondary workloads
def run_det(args, rank, world):
    """Secondary line: STTNDetInpaint on 46-frame 1080p batches (what `video_inpaint` feeds it for a 300-frame interval,
    batch_generator 46x6+24 — SURVEY §8a D-rows), device-resident and through the host call."""
    B, S = BACKEND, synthetic()
    eng, wdesc = make_sttn_det(B.device())
    T = 46
    frames = S.synthetic_clip(T, H, W, seed=100 + rank)
    mask = S.default_mask(H, W)
    stream = B.stream(eng.cuda_stream)
    work = [f.copy() for f in frames]
    warm = max(args.warmup, 3)
    for _ in range(warm):
        eng.stage(work, mask)
        eng.compute()
    eng.sync()
    evs = [(B.event(), B.event()) for _ in range(args.steps)]
    l0 = eng.launch_count
    B.barrier()
    B.sync()
    for a, b in evs:
        eng.stage(work, mask)
        eng.sync()
        a.record(stream)
        eng.compute()
        b.record(stream)
    eng.sync()
    B.sync()
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    launches = eng.launch_count - l0
    batches = [[f.copy() for f in frames] for _ in range(args.steps)]
    eng.inpaint_inplace([f.copy() for f in frames], mask)
    t0 = time.perf_counter()
    for b in batches:
        eng.inpaint_inplace(b, mask)
    e2e_s = time.perf_counter() - t0
    dev_ms, e2e_s = B.max_over_ranks([dev_ms, e2e_s])
    eng.stage(work, mask)
    eng.profile()
    eng.stage(work, mask)
    prof = eng.profile()
    conv_ms = prof["conv3x3"][0] + prof["conv3x3_residual"][0]
    passes = sum(len(nb) + len(rf) for nb, rf in chunk_schedule(T))
    conv_flop = 3 * 8 * passes * 60 * 108 * 2.0 * 2304 * 256
    burst, sustained, _, peak_src = peaks()
    if rank == 0:
        n = world * args.steps * T
        sh = int(W * 5 / 18)
        print(json.dumps({
            "metric": "inpainted frames/sec at 1080p (STTN-det, window=5)", "value": n / (dev_ms * 1e-3), "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": f"synthetic 1080p clip; {wdesc}",
            "config": {"workload": "STTN sttn-det inpaint on 46-frame 1080p batches (inpaint half of BASELINE config 4; detection not included)",
                       "frame": [H, W], "batch": T, "strip_h": sh},
            "e2e": {"value": n / e2e_s, "unit": "frames/s", "h2d_bytes_per_step": T * sh * W * 3, "d2h_bytes_per_step": T * sh * W * 3,
                    "api": "STTNDetInpaint.inpaint_inplace(frames, mask), synchronous"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "kernel": "tcgen05 implicit-GEMM 3x3 conv 256->256 on 60x108 maps, as it runs in the batch (in-situ events)",
                         "achieved": conv_flop / (conv_ms * 1e-3) / 1e12, "peak": sustained, "unit": "TFLOP/s",
                         "frac": conv_flop / (conv_ms * 1e-3) / 1e12 / sustained, "traffic": None, "peak_source": f"{peak_src} (sustained bf16)",
                         "in_situ_ms": {k: round(v[0], 3) for k, v in prof.items()},
                         "whole_step_frac_of_sustained": 758.2e9 * n / world / (dev_ms * 1e-3) / 1e12 / sustained}}), flush=True)


def _text_frames(n):
    import cv2

    yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
    frames = []
    for i in range(n):
        img = np.stack([96 + 60 * np.sin(xx / 211 + c + i) + 50 * np.cos(yy / 173 - c) for c in range(3)], -1).clip(0, 255).astype(np.uint8)
        for txt, org in ((f"The quick brown fox {i}123", (400, 1000)), ("second line of a subtitle", (500, 930))):
            cv2.putText(img, txt, org, cv2.FONT_HERSHEY_SIMPLEX, 2.0, (0, 0, 0), 9, cv2.LINE_AA)
            cv2.putText(img, txt, org, cv2.FONT_HERSHEY_SIMPLEX, 2.0, (255, 255, 255), 4, cv2.LINE_AA)
        frames.append(img)
    return frames


def run_dbnet(args, rank, world):
    """Secondary line: the DBNet text detector (SURVEY §8a T2) on 1080p frames — `SubtitleDetect.detect_subtitle`'s
    `TextDetection.predict` on the B200 against the oracle interpreter of the same PIR program on the host cores."""
    B = BACKEND
    frames = _text_frames(4)
    det = make_detector(B.device())
    warm = max(args.warmup, 3)
    for _ in range(warm):
        for f in frames:
            det.predict(f)
    per = 8
    B.barrier()
    B.sync()
    net_ms = det.time_network(args.steps * per)
    l0 = det.launch_count
    t0 = time.perf_counter()
    boxes = []
    for _ in range(args.steps):
        for j in range(per):
            boxes = det.predict(frames[j % len(frames)])[0]["dt_polys"]
    e2e_s = time.perf_counter() - t0
    net_ms, e2e_s = B.max_over_ranks([net_ms, e2e_s])
    cpu = None
    if rank == 0 and not args.no_cpu:
        import torch
        from oracle import dbnet_oracle as D

        g = D.Graph(detector_dir())
        D.detect_subtitle(g, frames[0])
        c0 = time.perf_counter()
        for f in frames[:3]:
            D.detect_subtitle(g, f)
        cpu = {"value": 3 / (time.perf_counter() - c0), "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": "3 of the 1080p frames through the oracle interpreter of the same PIR program (torch fp32) + DB post-process"}
    burst, sustained, _, peak_src = peaks()
    if rank == 0:
        n = world * args.steps * per
        flop = 267.6e9   # SURVEY §8d: 133.8 GMAC per [1,3,544,960] frame
        print(json.dumps({
            "metric": "text-detected frames/sec at 1080p (DBNet PP-OCRv5_server_det)", "value": world * 1e3 / net_ms, "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": net_ms * per, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16", "data": "synthetic 1080p frames with two rendered text lines; reference model files V5/ch_det",
            "config": {"workload": "DBNet detection of 1080p frames (detection half of BASELINE config 4): resize to 544x960, network, DB post-process",
                       "frame": [H, W], "frames_per_step": per, "boxes_last_frame": int(len(boxes))},
            "e2e": {"value": n / e2e_s, "unit": "frames/s", "h2d_bytes_per_step": per * H * W * 3, "d2h_bytes_per_step": per * 544 * 960 * 4,
                    "api": "TextDetector.predict(bgr_frame) -> dt_polys, synchronous, host post-process included"},
            "gpu_launches": int(args.steps * per * 247 + (det.launch_count - l0)),
            "roofline": {"bound": "tensor", "kernel": "whole network graph (247 launches, latency-bound small layers)", "achieved": flop / net_ms / 1e9,
                         "peak": sustained, "unit": "TFLOP/s", "frac": flop / net_ms / 1e9 / sustained, "traffic": None, "peak_source": f"{peak_src} (sustained bf16)"},
            "cpu_baseline": cpu}), flush=True)


def run_lama(args, rank, world):
    """Secondary line: LAMA (BASELINE config 1 / SURVEY §8a L1-L3) through `LamaInpaint.__call__` on 1080p frames: the strip
    of int(1920*3/16) = 360 rows around the subtitle goes through big-lama at native resolution, frame by frame."""
    B, S = BACKEND, synthetic()
    eng, wsrc, wdesc = make_lama(B.device())
    T = 4
    frames = S.synthetic_clip(T, H, W, seed=200 + rank)
    mask = S.default_mask(H, W)
    warm = max(args.warmup, 3)
    for _ in range(warm):
        eng(frames, mask)
    B.barrier()
    B.sync()
    net_ms = eng.model.time_network(args.steps * 2) / T      # one graph launch = the strips of T frames
    l0 = eng.model.launch_count
    t0 = time.perf_counter()
    for _ in range(args.steps):
        eng(frames, mask)
    e2e_s = time.perf_counter() - t0
    net_ms, e2e_s = B.max_over_ranks([net_ms, e2e_s])
    cpu = None
    if rank == 0 and not args.no_cpu:
        import torch
        from oracle import lama_oracle as LO

        w = LO.load_weights(wsrc)
        LO.lama_call(w, frames[:1], mask)
        c0 = time.perf_counter()
        LO.lama_call(w, frames[:2], mask)
        cpu = {"value": 2 / (time.perf_counter() - c0), "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": "2 of the 1080p frames through the oracle (torch fp32 restatement, bit-identical to the TorchScript module)"}
    burst, sustained, _, peak_src = peaks()
    if rank == 0:
        n = world * args.steps * T
        sh = int(W * 3 / 16)
        flop = 1158e9   # SURVEY §8d: conv FLOPs of one 360x1920 strip frame (+36 rfft2/irfft2 pairs)
        print(json.dumps({
            "metric": "inpainted frames/sec at 1080p (LAMA big-lama)", "value": world * 1e3 / net_ms, "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": net_ms * T, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16", "data": f"synthetic 1080p clip; {wdesc}",
            "config": {"workload": "LAMA inpaint of 1080p frames (BASELINE config 1 model on the video strip path): strip 360x1920 per frame",
                       "frame": [H, W], "frames_per_step": T, "strip_h": sh},
            "e2e": {"value": n / e2e_s, "unit": "frames/s", "h2d_bytes_per_step": T * (sh * W * 3 + sh * W), "d2h_bytes_per_step": T * sh * W * 3,
                    "api": "LamaInpaint.__call__(frames, mask), synchronous, copy semantics"},
            "gpu_launches": int(eng.model.launch_count - l0 + args.steps * 560),
            "roofline": {"bound": "tensor", "kernel": "whole network graph (~560 launches, 4 strips per launch, 45x240 feature grid)",
                         "achieved": flop / net_ms / 1e9, "peak": sustained, "unit": "TFLOP/s", "frac": flop / net_ms / 1e9 / sustained, "traffic": None,
                         "peak_source": f"{peak_src} (sustained bf16)"},
            "cpu_baseline": cpu}), flush=True)


def run_lama512(args, rank, world):
    """BASELINE config 1 itself: `LamaInpaint.inpaint(image, mask)` (lama_inpaint.py:17-28) on one 512x512 random-texture image with the
    rectangle mask rows 400-470, cols 60-450 (SURVEY §8d)."""
    B, S = BACKEND, synthetic()
    eng, wsrc, wdesc = make_lama(B.device())
    img = S.synthetic_clip(1, 512, 512, seed=0)[0]
    mask = np.zeros((512, 512), np.uint8)
    mask[400:470, 60:450] = 255
    warm = max(args.warmup, 3)
    for _ in range(warm):
        out = eng.inpaint(img, mask)
    B.barrier()
    B.sync()
    per = 8
    l0 = eng.model.launch_count
    t0 = time.perf_counter()
    for _ in range(args.steps * per):
        out = eng.inpaint(img, mask)
    e2e_s = time.perf_counter() - t0
    launches = eng.model.launch_count - l0
    net_ms = eng.model.time_network(args.steps * per)
    net_ms, e2e_s = B.max_over_ranks([net_ms, e2e_s])
    cpu = None
    if rank == 0 and not args.no_cpu:
        import torch
        from oracle import lama_oracle as LO

        w = LO.load_weights(wsrc)
        LO.inpaint(w, img, mask)
        c0 = time.perf_counter()
        LO.inpaint(w, img, mask)
        cpu = {"value": 1 / (time.perf_counter() - c0), "unit": "images/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": "the same 512x512 image through the oracle (torch fp32 restatement, bit-identical to the TorchScript module), once"}
    burst, sustained, _, peak_src = peaks()
    if rank == 0:
        n = world * args.steps * per
        flop = 439.8e9   # SURVEY §8a L2: conv FLOPs at 512x512
        print(json.dumps({
            "metric": "inpainted images/sec, LAMA 512x512 (BASELINE config 1)", "value": world * 1e3 / net_ms, "unit": "images/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": net_ms * per, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16", "data": f"synthetic 512x512 texture + rectangle mask; {wdesc}",
            "config": {"workload": "LAMA single-image inpaint 512x512 (BASELINE config 1)", "frame": [512, 512], "images_per_step": per,
                       "hole_mean": float(np.asarray(out)[400:470, 60:450].mean())},
            "e2e": {"value": n / e2e_s, "unit": "images/s", "h2d_bytes_per_step": per * (512 * 512 * 4), "d2h_bytes_per_step": per * 512 * 512 * 3,
                    "api": "LamaInpaint.inpaint(image, mask), synchronous"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "kernel": "whole network graph, one 64x64 feature grid (latency-bound: ~560 dependent launches)",
                         "achieved": flop / net_ms / 1e9, "peak": sustained, "unit": "TFLOP/s", "frac": flop / net_ms / 1e9 / sustained, "traffic": None,
                         "peak_source": f"{peak_src} (sustained bf16)"},
            "cpu_baseline": cpu}), flush=True)


def run_config4(args, rank, world):
    """BASELINE config 4 end to end on an in-memory 1080p clip: DBNet detection of the sampled frames -> interval planning ->
    create_mask -> STTN-det on batch_generator batches.  N = 1: `vsr_b200.video_inpaint_frames` (the loop of SubtitleRemover.video_inpaint,
    main.py:260-333).  N > 1 (`--gpus 8`, config 4's frame-batch shard): every rank detects its share of the sampled frames, ONE
    all_gather_object exchanges the hits, every rank plans identically and inpaints its share of the batches (vsr_b200.distributed)."""
    import cv2

    B, S = BACKEND, synthetic()
    T = 120 if world == 1 else 300
    frames = S.synthetic_clip(T, H, W, seed=300)          # the SAME clip on every rank: the job is sharded, not replicated (strong scaling)
    for i, f in enumerate(frames):                        # a subtitle on frames 11..T-10 (1-based), text changing every 48 frames
        if 10 <= i < T - 10:
            txt = f"subtitle line number {i // 48} of the clip"
            cv2.putText(f, txt, (420, 1020), cv2.FONT_HERSHEY_SIMPLEX, 1.8, (0, 0, 0), 9, cv2.LINE_AA)
            cv2.putText(f, txt, (420, 1020), cv2.FONT_HERSHEY_SIMPLEX, 1.8, (255, 255, 255), 4, cv2.LINE_AA)
    model, _ = make_sttn_det(B.device())
    det = make_subtitle_detect(B.device())
    det.SAMPLE_STEP = 3                                   # 30 fps video (subtitle_detect.py:29-39)
    if world == 1:
        from vsr_b200 import video_inpaint_frames

        run = lambda: video_inpaint_frames(frames, det, model)   # noqa: E731
    else:
        from vsr_b200.distributed import video_inpaint_frames_sharded

        run = lambda: video_inpaint_frames_sharded(frames, det, model, rank, world)   # noqa: E731
    warm = max(min(args.warmup, 2), 1)
    for _ in range(warm):
        out, sub, se = run()
    B.barrier()
    B.sync()
    l0 = model.launch_count
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out, sub, se = run()
    B.sync()
    B.barrier()
    e2e_s = time.perf_counter() - t0
    n_det = len(range(1, T + 1, 3))
    launches = model.launch_count - l0 + args.steps * (n_det // world) * 249   # + the detector's graph (247 kernels), pre-process, map extraction
    e2e_s, = B.max_over_ranks([e2e_s])
    n_inpainted = sum(e - s + 1 for s, e in se.items())
    if rank == 0:
        n = args.steps * T
        print(json.dumps({
            "metric": "frames/sec at 1080p, detection + STTN-det (BASELINE config 4)", "value": n / e2e_s, "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": e2e_s / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak" if world == 1 else "strong", "vs_baseline": None, "dtype": "f16",
            "data": "synthetic 1080p clip with rendered subtitles; reference model files",
            "config": {"workload": f"config 4 chain on a {T}-frame 1080p clip: DBNet on every 3rd frame, planning, create_mask, STTN-det batches"
                                   + ("" if world == 1 else f", sampled frames and batches dealt over {world} ranks, one all_gather_object of the detections"),
                       "frame": [H, W], "frames": T, "detected_frames": n_det, "inpainted_frames": n_inpainted,
                       "intervals": {str(k): v for k, v in se.items()}},
            "e2e": {"value": n / e2e_s, "unit": "frames/s", "h2d_bytes_per_step": n_det * H * W * 3 + n_inpainted * int(W * 5 / 18) * W * 3,
                    "d2h_bytes_per_step": n_inpainted * int(W * 5 / 18) * W * 3, "api": "vsr_b200.video_inpaint_frames(frames, SubtitleDetect, STTNDetInpaint)"},
            "gpu_launches": int(launches), "note": "host-timed whole chain (inputs are host numpy frames); the per-stage device numbers are the "
                                                   "sttn-det and dbnet workloads"}), flush=True)


def run_propainter(args, rank, world):
    """Secondary line: ProPainter (BASELINE config 3 / SURVEY §8a P1-P7) through `PropainterInpaint.__call__` on a 720p clip: the 240x1280
    strip around the subtitle goes through RAFT, flow completion, image propagation and the generator, `--pp-frames` frames per call
    (<= sub_video_length = 80, one reference sub-video).  There is no separate device-resident leg (flows take a host round trip between
    RAFT and the completion network): `value` is the same end-to-end rate."""
    B, S = BACKEND, synthetic()
    mdir = propainter_dir()
    Hp, Wp, T = 720, 1280, args.pp_frames
    frames = S.synthetic_clip(T, Hp, Wp, seed=300 + rank)
    mask = S.default_mask(Hp, Wp)
    eng = make_propainter(B.device())
    warm = max(args.warmup, 1)
    for _ in range(warm):
        eng(frames, mask)
    B.barrier()
    B.sync()
    sampler = ClockSampler(B.local)
    if rank == 0:
        sampler.start()
    l0 = eng._rt.launch_count
    t0 = time.perf_counter()
    for _ in range(args.steps):
        eng(frames, mask)
    B.sync()
    e2e_s = time.perf_counter() - t0
    launches = eng._rt.launch_count - l0
    clocks = sampler.stop() if rank == 0 else None
    e2e_s, = B.max_over_ranks([e2e_s])
    stages = getattr(eng, "stage_seconds", None)
    cpu = None
    if rank == 0 and not args.no_cpu:
        import torch
        from oracle import propainter_gen_oracle as G
        from oracle import raft_oracle as R
        from oracle import rfc_oracle as C

        w = {"raft": R.load_weights(os.path.join(mdir, "raft-things.pth")), "rfc": C.load_weights(os.path.join(mdir, "recurrent_flow_completion.pth")),
             "gen": G.load_weights(os.path.join(mdir, "ProPainter.pth"))}
        c0 = time.perf_counter()
        G.propainter_call(w, frames[:4], mask)
        cpu = {"value": 4 / (time.perf_counter() - c0), "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port",
               "sample": "4 of the 720p frames through the chained oracle (torch fp32 restatement, equal to the unmodified reference's frames)"}
    if rank == 0:
        from vsr_b200 import propainter_tools as PT

        (y0, y1, x0, x1), = PT.strip_areas(Wp, Hp, mask)
        sh, sw = y1 - y0, x1 - x0
        n = world * args.steps * T
        _, sustained, _, peak_src = peaks()
        flop = 2.52e12 * T      # SURVEY §8a: ~2.52 TFLOP per 720p frame (RAFT 1.35, generator 1.08, completion 0.10; measured at N = 12)
        print(json.dumps({
            "metric": "inpainted frames/sec at 720p (ProPainter)", "value": n / e2e_s, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": e2e_s / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16", "data": "synthetic 720p clip; reference ProPainter / RAFT / flow-completion weights",
            "config": {"workload": f"ProPainter on a {T}-frame 720p synthetic clip with optical-flow completion (BASELINE config 3, one sub-video per call)",
                       "frame": [Hp, Wp], "frames_per_step": T, "strip": [sh, sw], "l2": "inputs larger than L2 (strip frames + feature maps)"},
            "e2e": {"value": n / e2e_s, "unit": "frames/s", "h2d_bytes_per_step": T * sh * sw * 3 + sh * sw, "d2h_bytes_per_step": T * sh * sw * 3,
                    "api": "PropainterInpaint.__call__(frames, mask), synchronous, copy semantics"},
            "gpu_launches": int(launches), "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": "whole pipeline (RAFT + flow completion + propagation + generator), host-timed",
                         "achieved": flop * args.steps / e2e_s / 1e12, "peak": sustained, "unit": "TFLOP/s",
                         "frac": flop * args.steps / e2e_s / 1e12 / sustained, "traffic": None, "peak_source": f"{peak_src} (sustained bf16)",
                         "stage_seconds_last_call": stages},
            "cpu_baseline": cpu}), flush=True)


def run_sttn_strong(args, rank, world):
    """Single-clip strong scaling (SURVEY §8e): ONE 300-frame 1080p clip (BASELINE config 2's clip), chunk by chunk, every chunk's windows
    dealt over all `world` GPUs (`STTNInpaint.inpaint_chunk_sharded`: NCCL all-gather of the reference-frame encoder features and of the
    window predictions, blend replayed in schedule order — output bit-identical to one GPU).  Host frames in, result strips in host memory
    on the rank that owns each frame; wall clock, max over ranks."""
    B, S = BACKEND, synthetic()
    eng, src, wdesc = make_sttn(B.device())
    n_chunks = 6
    frames = S.synthetic_clip(CHUNK, H, W, seed=0)      # the same clip on every rank: the job is sharded, not replicated
    mask = S.default_mask(H, W)
    warm = max(min(args.warmup, 3), 1)
    for _ in range(warm):
        eng.inpaint_chunk_sharded([f.copy() for f in frames], mask, rank, world)
    vals = []
    for _ in range(args.steps):
        clips = [[f.copy() for f in frames] for _ in range(n_chunks)]
        l0 = eng.launch_count
        B.barrier()
        B.sync()
        t0 = time.perf_counter()
        for c in clips:
            eng.inpaint_chunk_sharded(c, mask, rank, world)
        B.sync()
        B.barrier()
        vals.append(time.perf_counter() - t0)
        launches = eng.launch_count - l0
    e2e_s, = B.max_over_ranks([float(np.sum(vals))])
    if rank == 0:
        n = args.steps * n_chunks * CHUNK
        sh = int(W * 3 / 16)
        _, sustained, _, peak_src = peaks()
        fpix = 30 * 160 * 256
        print(json.dumps({
            "metric": METRIC, "value": n / e2e_s, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": e2e_s / args.steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f16",
            "data": f"synthetic 1080p clip (seeded, generated on host); {wdesc}",
            "config": {"workload": "ONE 300-frame 1080p clip (6 chunks of 50), every chunk's 10 windows dealt over the ranks, reference-frame "
                                   "features and window predictions all-gathered over NVLink (single-clip latency, BASELINE config 2's clip)",
                       "frame": [H, W], "chunk": CHUNK, "frames_per_step": n_chunks * CHUNK, "neighbor_stride": 5, "ref_length": 10,
                       "parallelism": f"window-per-rank x{world}",
                       "collective_bytes_per_chunk": {"reference_features": 5 * fpix * 6, "window_predictions": 10 * 32 * 120 * 640 * 3 * 4}},
            "e2e": {"value": n / e2e_s, "unit": "frames/s", "h2d_bytes_per_step": n_chunks * CHUNK * sh * W * 3,
                    "d2h_bytes_per_step": n_chunks * ((CHUNK + world - 1) // world) * sh * W * 3,
                    "api": "STTNInpaint.inpaint_chunk_sharded(frames, mask, rank, world) per chunk, synchronous (every rank uploads the chunk's strips)"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "kernel": "whole clip, all ranks (eager launches, no CUDA graph in the sharded path)",
                         "achieved": FLOP_PER_FRAME * n / e2e_s / 1e12, "peak": sustained * world, "unit": "TFLOP/s",
                         "frac": FLOP_PER_FRAME * n / e2e_s / 1e12 / (sustained * world), "traffic": None, "peak_source": f"{peak_src} (sustained bf16 x ranks)"}}),
            flush=True)


def ncu_traffic():
    """dram bytes per launch of the dominant kernel from the committed `ncu --set full` capture (tools/ncu_summary.py writes it)."""
    p = os.path.join(ROOT, "profiles", "ncu_r2_conv3x3.json")
    try:
        d = json.load(open(p))
        return float(d["dram_bytes_per_launch"]), os.path.relpath(p, ROOT)
    except Exception:
        return None, None


def settle_attention_path(eng, frames, mask):
    """One checked pass of the chunk, the check every call of STTNInpaint makes: when the chunk's attention logits leave the range of the
    single-pass softmax (attn_direct), the frames of that pass are rejected and the engine switches to the score matrix + softmax kernel
    for good (STTNInpaint._exact_softmax_retry).  The unchecked passes timed after it then compute the frames a caller receives (the
    seeded random-init weights take every 1080p pass of the chunk out of that range).  Returns the name of the path."""
    from vsr_b200._capi import VsrRangeError

    eng.stage(frames, mask)
    eng.compute()
    try:
        eng.fetch([np.empty_like(f) for f in frames])
        return "single-pass softmax"
    except VsrRangeError:
        eng.set_option("attn_direct", 0)
        return "score matrix + softmax kernel (logits beyond the single-pass range)"


DUMP_PIXELS = {"inpainted": 1 << 16, "kept": 1 << 14}   # 50 frames x (65536 + 16384) pixels x 3 channels x 4 bytes = 49 MB


def output_sample(frames, mask, seed=0):
    """A fixed, seeded sample of a chunk's output frames (50 x 1080p = 311 MB, too large to store whole): float32 [T, n, 3] at the same
    pixel positions in every frame, "inpainted" under the mask (where the network's prediction is composited) and "kept" outside it
    (copied from the input)."""
    rng = np.random.default_rng(seed)
    under = np.asarray(mask).reshape(-1) != 0
    out = {}
    for name, where in (("inpainted", under), ("kept", ~under)):
        idx = np.flatnonzero(where)
        idx = np.sort(rng.choice(idx, min(DUMP_PIXELS[name], idx.size), replace=False))
        out[name] = np.stack([f.reshape(-1, 3)[idx] for f in frames]).astype(np.float32)
    return out


def write_outputs(path, arrays):
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------ the contract line: sttn-auto
def run_sttn_auto(args, rank, world):
    B, S = BACKEND, synthetic()
    eng, src, wdesc = make_sttn(B.device())
    frames = S.synthetic_clip(CHUNK, H, W, seed=rank)  # each rank its own chunk (weak scaling)
    mask = S.default_mask(H, W)
    stream = B.stream(eng.cuda_stream)
    strip_bytes = CHUNK * int(W * 3 / 16) * W * 3
    warm = max(args.warmup, 3)

    # ---- device-resident leg: strips staged once, K timed chunk passes ------------------------
    work = [f.copy() for f in frames]
    attention = settle_attention_path(eng, work, mask)
    eng.stage(work, mask)
    for _ in range(warm):
        eng.stage(work, mask)  # restore the original strips (compute composites in place)
        eng.compute()
    eng.sync()
    sampler = ClockSampler(B.local)
    if rank == 0:
        sampler.start()
    evs = [(B.event(), B.event()) for _ in range(args.steps)]
    launches0 = eng.launch_count
    B.barrier()
    B.sync()
    for i in range(args.steps):
        eng.stage(work, mask)   # untimed: H2D of the strips (the timed region starts with inputs in HBM)
        eng.sync()
        evs[i][0].record(stream)
        eng.compute()
        evs[i][1].record(stream)
    eng.sync()
    B.sync()
    B.barrier()
    launches = eng.launch_count - launches0
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    dev_ms, = B.max_over_ranks([dev_ms])
    dumped = None
    if args.dump_outputs and rank == 0:     # before the legs below reuse the engine: the frames of the last timed step
        outs = [np.empty_like(f) for f in frames]
        eng.fetch(outs)
        dumped = output_sample(outs, mask)
        del outs

    # ---- end-to-end leg: host numpy frames in, host numpy frames out --------------------------
    # (a) the chunk loop of STTNAutoInpaint.__call__: two chunks in flight (submit / collect), every step
    #     still pays its own host->pinned copy, H2D, kernels, D2H and pinned->host copy
    for _ in range(2):
        eng.inpaint_inplace([f.copy() for f in frames], mask)
    warm_batches = [[f.copy() for f in frames] for _ in range(4)]  # warm both pipeline slots (pinned buffers, graph re-capture)
    prev = None
    for b in warm_batches:
        ticket = eng.submit(b, mask)
        if prev is not None:
            eng.collect(prev[0], prev[1])
        prev = (ticket, b)
    eng.collect(prev[0], prev[1])
    del warm_batches
    batches = [[f.copy() for f in frames] for _ in range(args.steps)]
    B.barrier()
    B.sync()
    t0 = time.perf_counter()
    prev = None
    for b in batches:
        ticket = eng.submit(b, mask)
        if prev is not None:
            eng.collect(prev[0], prev[1])
        prev = (ticket, b)
    eng.collect(prev[0], prev[1])
    e2e_s = time.perf_counter() - t0
    # (b) strictly synchronous calls, one chunk at a time
    batches = [[f.copy() for f in frames] for _ in range(args.steps)]
    t0 = time.perf_counter()
    for b in batches:
        eng.inpaint_inplace(b, mask)
    e2e_sync_s = time.perf_counter() - t0
    e2e_s, e2e_sync_s = B.max_over_ranks([e2e_s, e2e_sync_s])
    clocks = sampler.stop() if rank == 0 else None

    # ---- roofline of the dominant kernel, in situ -----------------------------------------------
    # One eager pass of the same chunk with events around every launch group (the second of two, so that nothing allocates).
    eng.stage(work, mask)
    eng.profile()
    eng.stage(work, mask)
    prof = eng.profile()
    conv_ms = prof["conv3x3"][0] + prof["conv3x3_residual"][0]
    conv_launches = prof["conv3x3"][1] + prof["conv3x3_residual"][1]
    passes = sum(len(nb) + len(rf) for nb, rf in chunk_schedule(CHUNK))           # 140 frame-passes per 50-frame chunk (SURVEY §8a A6)
    conv_flop = 3 * 8 * passes * 30 * 160 * 2.0 * 2304 * 256                       # 3 convs x 8 blocks, 2*9*256*256 FLOP per pixel
    prof_total = sum(v[0] for v in prof.values())
    group = int(os.environ.get("VSR_WINDOW_GROUP", "2"))
    Tw = 29 if group >= 2 else 15  # frames per conv launch in the steady state (windows of 15 + 14 share a launch)
    iso_ms = float(np.median(eng.time_conv(Tw, 20)))
    iso_flop = 2.0 * Tw * 30 * 160 * 2304 * 256
    burst, sustained, hbm, peak_src = peaks()
    traffic, traffic_src = ncu_traffic()
    achieved = conv_flop / (conv_ms * 1e-3) / 1e12
    roof = {"bound": "tensor",
            "kernel": "tcgen05 implicit-GEMM 3x3 conv 256->256 on 30x160 maps (transformer blocks: output_linear, feed_forward.conv.0/.2), "
                      "as it runs in the chunk: CUDA events around each of its launches in one eager pass of the timed chunk",
            "achieved": achieved, "peak": sustained, "unit": "TFLOP/s", "frac": achieved / sustained,
            "traffic": traffic, "traffic_source": traffic_src, "peak_source": f"{peak_src} (sustained bf16: kernel timed inside a long step)",
            "launches": int(conv_launches), "ms_per_launch": conv_ms / max(conv_launches, 1), "flop_per_launch": conv_flop / max(conv_launches, 1),
            "share_of_step": conv_ms / prof_total if prof_total else None,
            "in_situ_ms": {k: round(v[0], 3) for k, v in prof.items()},
            "isolated": {"what": f"same kernel, LeakyReLU epilogue only, {Tw} frames, 20 back-to-back launches on the same buffers (L2-warm)",
                         "achieved": iso_flop / (iso_ms * 1e-3) / 1e12, "frac_of_burst": iso_flop / (iso_ms * 1e-3) / 1e12 / burst, "peak_burst": burst},
            "whole_step_frac_of_sustained": (FLOP_PER_FRAME * CHUNK * args.steps / (dev_ms * 1e-3)) / 1e12 / sustained}

    if rank != 0:
        return

    # ---- CPU baseline on a bounded sample (rank 0, N = 1 only) ---------------------------------
    cpu = None
    if world == 1 and not args.no_cpu:
        cpu = cpu_baseline_leg(src, frames, mask, args.cpu_frames)

    total_frames = world * args.steps * CHUNK
    line = {"metric": METRIC, "value": total_frames / (dev_ms * 1e-3), "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16", "data": f"synthetic 1080p clip (seeded, generated on host); {wdesc}",
            "config": {"workload": WORKLOAD, "frame": [H, W], "chunk": CHUNK, "neighbor_stride": 5, "ref_length": 10, "strip": [720, 1080, 0, 1920],
                       "l2": "per-step working set (104 MB strips + ~0.9 GB activations) exceeds the 126 MB L2", "attention": attention,
                       "parallelism": f"chunk-per-rank x{world}" if world > 1 else "single GPU"},
            "e2e": {"value": total_frames / e2e_s, "unit": "frames/s", "h2d_bytes_per_step": strip_bytes,
                    "d2h_bytes_per_step": strip_bytes,
                    "api": "STTNInpaint.submit/collect on numpy frames (the chunk loop of STTNAutoInpaint.__call__, two chunks in flight)",
                    "sync_value": total_frames / e2e_sync_s, "sync_api": "STTNInpaint.inpaint_inplace(frames, mask), one chunk at a time"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu}
    print(json.dumps(line), flush=True)
    if dumped is not None:
        write_outputs(args.dump_outputs, dumped)


WORKLOADS = {"sttn-auto": run_sttn_auto, "sttn-auto-strong": run_sttn_strong, "sttn-det": run_det, "dbnet": run_dbnet, "lama": run_lama, "lama512": run_lama512, "config4": run_config4,
             "propainter": run_propainter}


def main(argv=None):
    global BACKEND
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--cpu-frames", type=int, default=32, help="frames of the chunk the cpu_baseline leg runs through the reference (<= 50)")
    ap.add_argument("--workload", default="sttn-auto", choices=sorted(WORKLOADS),
                    help="sttn-auto = BASELINE config 2 (the contract line); sttn-det / dbnet = the inpaint / detection halves of config 4; "
                         "config4 = that chain end to end (sharded over the ranks when N > 1); lama = the big-lama model of config 1 on 1080p "
                         "strips; lama512 = config 1 itself; propainter = config 3")
    ap.add_argument("--pp-frames", type=int, default=40, help="frames per call of the propainter workload (<= 80)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the frames the last timed step computed to DIR/*.npy "
                                                          "(float32, 49 MB; sttn-auto workload)")
    args = ap.parse_args(argv)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "sttn-auto"):
        ap.error("--dump-outputs is implemented for --impl b200 --workload sttn-auto")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    if BACKEND is None:
        BACKEND = CudaBackend()
    if not BACKEND.available():
        raise SystemExit("bench.py needs a B200: vsr_b200 has no CPU fallback")
    BACKEND.setup(local, world)
    try:
        WORKLOADS[args.workload](args, rank, world)
    finally:
        BACKEND.finish()


if __name__ == "__main__":
    main()
