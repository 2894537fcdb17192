"""CPU dry run of bench.py: every workload and both arms run `bench.main()` with stand-ins for CUDA (bench.BACKEND) and for the engines
(the bench.make_* factories), so that a name error, a broken unpacking or a JSON-schema regression in the contract line fails here, in
`-m "not gpu"`, and not on the driver's GPU box at the end of a round.  Only the *plumbing* of bench.py is exercised; numbers are fake."""
import json
import time

import numpy as np
import pytest

import bench
from vsr_b200._capi import VsrRangeError


class _Event:
    def __init__(self):
        self.t = None

    def record(self, stream=None):
        self.t = time.perf_counter()

    def elapsed_time(self, other):
        return max((other.t - self.t) * 1e3, 1e-3)


class FakeBackend:
    local, world = 0, 1

    def available(self):
        return True

    def setup(self, local, world):
        self.local, self.world = local, world

    def device(self):
        return "cuda:0"

    def sync(self):
        pass

    def barrier(self):
        pass

    def event(self):
        return _Event()

    def stream(self, ptr):
        return None

    def max_over_ranks(self, values):
        return [float(v) for v in values]

    def finish(self):
        pass


class FakeSTTN:
    """duck type of vsr_b200.STTNInpaint / STTNDetInpaint as bench.py uses it"""
    PROF = ("conv3x3", "conv3x3_residual", "qkv", "score", "softmax", "pv", "encoder", "decoder", "gather", "prepost")
    cuda_stream = 0

    def __init__(self, out_of_range=False):
        self.launch_count = 0
        self.tickets = 0
        self.computes = 0
        self.out_of_range = out_of_range    # logits beyond the single-pass softmax: fetch raises until attn_direct is switched off
        self.options = {"attn_direct": 1}

    def set_option(self, name, value):
        self.options[name] = value

    def stage(self, frames, mask):
        assert frames[0].dtype == np.uint8 and mask.shape == frames[0].shape[:2]
        self.staged = (frames, mask)

    def compute(self):
        self.launch_count += 700
        self.computes += 1
        time.sleep(0.001)

    def fetch(self, frames_out):
        """the staged frames with the number of compute() calls so far written under the mask"""
        if self.out_of_range and self.options["attn_direct"]:
            raise VsrRangeError("attention logits beyond the range of the single-pass softmax (attn_direct)")
        frames, mask = self.staged
        for o, f in zip(frames_out, frames):
            o[...] = f
            o[mask != 0] = self.computes

    def sync(self):
        pass

    def inpaint_inplace(self, frames, mask):
        self.launch_count += 700

    def inpaint_chunk_sharded(self, frames, mask, rank, world):
        self.launch_count += 700
        return list(range(rank, len(frames), world))

    def submit(self, frames, mask):
        self.tickets += 1
        return self.tickets

    def collect(self, ticket, frames):
        pass

    def profile(self):
        return {k: (1.0 + i, 10 * (i + 1)) for i, k in enumerate(self.PROF)}

    def time_conv(self, T, n):
        return np.full(n, 0.1, np.float32)

    def __call__(self, frames, mask):
        self.launch_count += 700
        return [f.copy() for f in frames]


class FakeDetector:
    launch_count = 0

    def predict(self, img):
        return [{"dt_polys": [np.zeros((4, 2))]}]

    def time_network(self, n):
        return 3.0


class FakeSubtitleDetect:
    SAMPLE_STEP = 3

    def scan_frames(self, frames, sections=None, on_frame=None):
        return {i: [(420, 1500, 960, 1040)] for i in range(11, len(frames) - 9)}


class FakeLama:
    class model:
        launch_count = 0

        @staticmethod
        def time_network(n):
            return 20.0

    def __call__(self, frames, mask):
        return [f.copy() for f in frames]

    def inpaint(self, img, mask):
        return np.asarray(img).copy()


class FakePropainter:
    class _rt:
        launch_count = 0

    stage_seconds = {"raft": 0.1}

    def __call__(self, frames, mask):
        return [f.copy() for f in frames]


CONTRACT_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
                 "data", "config", "e2e", "gpu_launches"}


@pytest.fixture
def fake_world(monkeypatch, tmp_path):
    monkeypatch.setattr(bench, "BACKEND", FakeBackend())
    monkeypatch.setattr(bench, "make_sttn", lambda dev: (FakeSTTN(), {"w": np.zeros(1, np.float32)}, "stand-in weights"))
    monkeypatch.setattr(bench, "make_sttn_det", lambda dev: (FakeSTTN(), "stand-in weights"))
    monkeypatch.setattr(bench, "make_detector", lambda dev: FakeDetector())
    monkeypatch.setattr(bench, "make_subtitle_detect", lambda dev: FakeSubtitleDetect())
    monkeypatch.setattr(bench, "make_lama", lambda dev: (FakeLama(), "none.npz", "stand-in weights"))
    monkeypatch.setattr(bench, "make_propainter", lambda dev: FakePropainter())
    monkeypatch.setattr(bench, "propainter_dir", lambda: str(tmp_path))
    monkeypatch.setattr(bench, "detector_dir", lambda: str(tmp_path))
    monkeypatch.setattr(bench.ClockSampler, "start", lambda self: None)
    monkeypatch.setattr(bench.ClockSampler, "stop", lambda self: {"sm_mhz": 1800.0, "sm_max_mhz": 1965.0, "reasons": [], "samples": 3})
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        monkeypatch.delenv(k, raising=False)


def _line(capsys):
    out = [ln for ln in capsys.readouterr().out.splitlines() if ln.startswith("{")]
    assert len(out) == 1, out
    return json.loads(out[0])


@pytest.mark.parametrize("workload", sorted(bench.WORKLOADS))
def test_every_workload_prints_one_contract_line(fake_world, capsys, workload):
    bench.main(["--workload", workload, "--steps", "2", "--warmup", "1", "--no-cpu", "--pp-frames", "4"])
    d = _line(capsys)
    assert CONTRACT_KEYS <= set(d), CONTRACT_KEYS - set(d)
    assert d["value"] > 0 and d["e2e"]["value"] > 0 and d["steps"] == 2 and d["higher_is_better"] is True
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"]) and d["e2e"]["h2d_bytes_per_step"] > 0
    assert "workload" in d["config"] and "model" not in d["config"]
    if workload != "config4":
        assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(d["roofline"])
        assert abs(d["roofline"]["frac"] - d["roofline"]["achieved"] / d["roofline"]["peak"]) < 1e-9


def test_contract_line_with_cpu_baseline(fake_world, capsys, monkeypatch):
    """the default invocation (N = 1, cpu_baseline leg included) down to the last key the driver reads"""
    calls = []

    class FakeCpu:
        kind, threads = "reference", 8

        def __init__(self, src, threads=None):
            calls.append(src)

        def fps(self, frames, mask):
            return 1.25, len(frames) / 1.25

        def pick_threads(self, frames, mask):
            return 1.25

        def describe(self):
            return "stand-in"

    monkeypatch.setattr(bench, "CpuReference", FakeCpu)
    bench.main(["--gpus", "1", "--steps", "3", "--warmup", "3"])
    d = _line(capsys)
    assert d["metric"] == bench.METRIC and d["unit"] == "frames/s" and d["n_gpus"] == 1 and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["dtype"] == "f16" and d["gpu_launches"] == 3 * 700
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] == 8 and d["cpu_baseline"]["value"] == 1.25 and calls
    r = d["roofline"]
    assert r["bound"] == "tensor" and r["unit"] == "TFLOP/s" and r["launches"] == 30 and set(r["in_situ_ms"]) == set(FakeSTTN.PROF)
    assert d["clocks"]["sm_mhz"] == 1800.0


def test_dump_outputs_of_the_last_timed_step(fake_world, capsys, tmp_path):
    """--dump-outputs: float32 samples of the frames fetched after the last of --steps timed steps, within 64 MB, equal from run to run"""
    runs = []
    for k in range(2):
        bench.main(["--steps", "4", "--warmup", "3", "--no-cpu", "--dump-outputs", str(tmp_path / str(k))])
        d = _line(capsys)
        assert d["steps"] == 4 and d["config"]["attention"] == "single-pass softmax"
        runs.append({p.stem: np.load(p) for p in (tmp_path / str(k)).glob("*.npy")})
    a, b = runs
    assert set(a) == {"inpainted", "kept"} and all(v.dtype == np.float32 and v.shape[:1] == (bench.CHUNK,) for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert all(np.array_equal(a[k], b[k]) for k in a)
    assert np.all(a["inpainted"] == 1 + 3 + 4)                      # fetched after the checked pass, the 3 warm-up and the 4 timed computes
    S = bench.synthetic()
    want = bench.output_sample(S.synthetic_clip(bench.CHUNK, bench.H, bench.W, seed=0), S.default_mask(bench.H, bench.W))
    assert np.array_equal(a["kept"], want["kept"])                  # outside the mask: the input frames
    for bad in (["--steps", "0"], ["--workload", "lama", "--dump-outputs", str(tmp_path)]):
        with pytest.raises(SystemExit):
            bench.main(bad)


def test_timed_path_is_the_one_a_caller_gets_when_logits_leave_the_single_pass_range(fake_world, capsys, monkeypatch, tmp_path):
    """a chunk the single-pass softmax cannot hold: its results are rejected, so the timed steps run (and the dump reads) the exact path"""
    eng = FakeSTTN(out_of_range=True)
    monkeypatch.setattr(bench, "make_sttn", lambda dev: (eng, {"w": np.zeros(1, np.float32)}, "stand-in weights"))
    bench.main(["--steps", "2", "--warmup", "1", "--no-cpu", "--dump-outputs", str(tmp_path)])
    assert _line(capsys)["config"]["attention"].startswith("score matrix + softmax kernel") and eng.options["attn_direct"] == 0
    assert np.all(np.load(tmp_path / "inpainted.npy") == 1 + 3 + 2)


def test_reference_arm_line(capsys, monkeypatch):
    class FakeCpu:
        kind, threads = "port", 4

        def __init__(self, src, threads=None):
            pass

        def fps(self, frames, mask):
            return 2.0, len(frames) / 2.0

        def pick_threads(self, frames, mask):
            return 2.0

        def describe(self):
            return "stand-in"

    monkeypatch.setattr(bench, "CpuReference", FakeCpu)
    monkeypatch.setattr(bench, "CPU_BUDGET_S", 30.0)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        monkeypatch.delenv(k, raising=False)
    bench.main(["--impl", "reference", "--gpus", "1", "--steps", "20", "--warmup", "5"])
    d = _line(capsys)
    assert d["impl"] == "reference" and d["metric"] == bench.METRIC and d["unit"] == "frames/s" and abs(d["value"] - 2.0) < 1e-9
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"] and d["config"]["frames_per_step"] in bench.CPU_SAMPLE_SIZES
    # ranks other than 0 print nothing and exit 0
    monkeypatch.setenv("RANK", "1")
    monkeypatch.setenv("WORLD_SIZE", "2")
    bench.main(["--impl", "reference", "--gpus", "2", "--steps", "2", "--warmup", "1"])
    assert capsys.readouterr().out.strip() == ""


def test_cpu_reference_runs_the_unmodified_reference_or_the_port():
    """CpuReference on a tiny clip: kind "reference" when the reference modules are present (baseline/_ref or /root/reference), else the port;
    both return frames of the input shape."""
    import os

    from vsr_b200 import synthetic as S

    p = os.path.join(bench.ROOT, "weights", "sttn-auto", "infer_model.pth")
    src = p if os.path.exists(p) else S.random_sttn_weights(0)
    cpu = bench.CpuReference(src, threads=4)
    frames = S.synthetic_clip(3, 135, 240, seed=1)
    out = cpu(frames, S.default_mask(135, 240))
    assert len(out) == 3 and out[0].shape == frames[0].shape and out[0].dtype == np.uint8
    assert cpu.kind == ("reference" if isinstance(src, str) and bench.reference_available() else "port")


def test_sample_sizing():
    class Quad:      # a CPU whose call costs 0.05 s per frame squared
        def fps(self, frames, mask):
            return 1.0, 0.05 * len(frames) ** 2

    frames = list(range(50))
    assert bench.cpu_sample_frames(Quad(), frames, None, 9.6) == 10          # 6 -> 1.8 s, 10 -> 5 s, 16 predicted 12.8 s <= 14.4: tried, 12.8 s > budget
    assert bench.cpu_sample_frames(Quad(), frames, None, 1000.0) == 50 and bench.cpu_sample_frames(Quad(), frames, None, 0.1) == 6
    assert sum(len(a) + len(b) for a, b in bench.chunk_schedule(50)) == 140      # SURVEY §8a A6
