"""bench.py contract on CPU: the reference arm (`--impl reference`) prints ONE JSON line with the keys the driver
reads, rank != 0 prints nothing, and the GPU arm refuses to run without a B200 (no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=300,
                          env=dict(os.environ, **(env or {})))


def test_reference_arm_json_line():
    r = _run(["--impl", "reference", "--workload", "tiny", "--steps", "1", "--warmup", "0", "--ref-prompt-len", "8", "--ref-new-tokens", "3"])
    assert r.returncode == 0, r.stderr[-500:]
    lines = [l for l in r.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "decode_tokens_per_sec" and d["unit"] == "tokens/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["ms_per_step"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert d["e2e"] == {"value": d["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_falcon_family():
    """BASELINE config 4 is a Falcon model: the CPU arm must build that family too (FalconForCausalLM, eager)."""
    r = _run(["--impl", "reference", "--workload", "tiny-falcon", "--steps", "1", "--warmup", "0", "--ref-prompt-len", "8", "--ref-new-tokens", "3"])
    assert r.returncode == 0, r.stderr[-800:]
    d = json.loads([l for l in r.stdout.strip().splitlines() if l.startswith("{")][0])
    assert d["impl"] == "reference" and d["value"] > 0 and "tiny-falcon" in d["config"]["workload"]


def test_reference_arm_other_ranks_are_silent():
    r = _run(["--impl", "reference", "--workload", "tiny", "--gpus", "2"], env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_gpu_arm_refuses_without_a_gpu():
    if torch.cuda.is_available():
        import pytest

        pytest.skip("GPU present")
    r = _run(["--workload", "tiny", "--steps", "1", "--warmup", "0"])
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_gpu_arm_control_flow_against_a_mock_engine(monkeypatch, capsys, tmp_path):
    """bench.py's GPU arm end to end on CPU with a mock Engine (control flow and JSON contract, not numbers): the keys the
    driver reads, the TTFT top-up to >= 20 samples (SURVEY.md 8d), a failing batch-32 sub-measurement that must not lose
    the headline line, --engine-params echoed in config, --dump-outputs writing the ids of the last timed request."""
    import importlib
    import time

    import numpy as np

    import substratus_b200

    class Timing:
        prefill_ms, decode_ms, kernel_launches, h2d_bytes, d2h_bytes = 1.0, 2.0, 129, 4096, 512

    class Info:
        weight_bytes_per_step, kv_bytes_per_token, hbm_bytes_allocated, hidden_size = 13.2e9, 524288, 14e9, 4096

    class MockEngine:
        def __init__(self, model_dir, params):
            self.info, self.params, self.n, self.calls = Info(), params, 0, 0

        def seq_create(self):
            self.n += 1
            return self.n

        def seq_free(self, sid):
            pass

        def prefill(self, sids, prompts):
            if self.params.get("fail32") and len(sids) == 32:
                raise RuntimeError("boom")
            time.sleep(0.001)
            self.calls += 1  # ids tell the requests apart
            return np.full(len(sids), self.calls, dtype=np.int32), None

        def decode(self, sids, first, n):
            time.sleep(0.002)
            return np.tile(np.arange(n, dtype=np.int32), (len(sids), 1)) + first[:, None], None

        def timing(self):
            return Timing()

        def timing_reset(self):
            pass

        def bench_kernel(self, kind, rows, ctx, iters):
            return 0.03, 1.8e8

        def close(self):
            pass

    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(torch.cuda, "set_device", lambda d: None)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    monkeypatch.setattr(substratus_b200, "Engine", MockEngine)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        monkeypatch.delenv(k, raising=False)
    sys.path.insert(0, ROOT)
    bench = importlib.import_module("bench")

    def run(argv):
        monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
        capsys.readouterr()
        bench.main()
        lines = [l for l in capsys.readouterr().out.splitlines() if l.startswith("{")]
        assert len(lines) == 1  # ONE JSON line
        return json.loads(lines[0])

    d = run(["--steps", "3", "--warmup", "1", "--no-cpu-baseline", "--no-extras"])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
                "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "ttft_ms_p50"):
        assert key in d, key
    assert d["steps"] == 3 and d["n_gpus"] == 1 and d["ttft_samples"] == 20 and d["batch32"]["value"] > 0
    assert set(d["e2e"]) >= {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"}
    assert set(d["roofline"]) >= {"bound", "achieved", "peak", "unit", "frac", "traffic"} and d["roofline"]["kernel"].startswith("decode_mega_kernel")
    d = run(["--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--no-extras", "--engine-params", '{"fail32": 1}'])
    assert d["value"] > 0 and "boom" in d["batch32"]["error"] and d["config"]["engine_params"] == {"fail32": 1}
    d = run(["--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--no-extras", "--batch", "32"])
    assert d["config"]["batch"] == 32 and "batch32" not in d and d["roofline"]["kernel"].startswith("gate/up")
    d = run(["--steps", "25", "--warmup", "1", "--no-cpu-baseline", "--no-batch32", "--no-extras"])
    assert d["ttft_samples"] == 25
    out = tmp_path / "outputs"
    run(["--steps", "3", "--warmup", "2", "--batch", "2", "--no-cpu-baseline", "--no-batch32", "--no-extras", "--dump-outputs", str(out)])
    assert sorted(os.listdir(out)) == ["decode_tokens.npy", "prefill_tokens.npy"]
    pre, dec = np.load(out / "prefill_tokens.npy"), np.load(out / "decode_tokens.npy")
    assert pre.dtype == dec.dtype == np.float32 and pre.shape == (2,) and dec.shape == (2, bench.NEW_TOKENS - 1)
    assert (pre == 5).all()  # prefill call 5 = the third timed request after two warm-ups, not a later TTFT top-up
    assert (dec == 5 + np.arange(bench.NEW_TOKENS - 1)).all()
    with pytest.raises(SystemExit):
        run(["--steps", "0", "--no-cpu-baseline", "--no-extras"])


def test_reference_arm_is_a_full_depth_measurement():
    """VERDICT r1 item 7: no layer extrapolation — the line describes exactly what was timed."""
    r = _run(["--impl", "reference", "--workload", "tiny", "--steps", "3", "--warmup", "1", "--ref-prompt-len", "16", "--ref-new-tokens", "4"])
    assert r.returncode == 0, r.stderr[-500:]
    d = json.loads([l for l in r.stdout.strip().splitlines() if l.startswith("{")][0])
    assert d["steps"] == 3 and d["tokens_per_step"] >= 1 and "full-depth (8 layers" in d["config"]["sample"] and "extrapolat" not in d["config"]["sample"]
    assert abs(d["value"] - d["tokens_per_step"] * 1e3 / d["ms_per_step"]) / d["value"] < 1e-6  # value == tokens per step / mean step time


def test_synthetic_q4_0_gguf_writer(tmp_path):
    """bench.py's config-3 file generator: a well-formed Q4_0 GGUF the engine's own reader accepts (host side only)."""
    import importlib

    sys.path.insert(0, ROOT)
    bench = importlib.import_module("bench")
    from substratus_b200.engine import model_read_tensor, model_tensor_count

    cfg = dict(bench.WORKLOADS["tiny"], num_hidden_layers=2, intermediate_size=704)
    size = bench.write_q4_0_gguf(str(tmp_path / "model.bin"), cfg)
    assert size > 0 and model_tensor_count(str(tmp_path)) == 3 + 9 * 2
    dt, shape, raw = model_read_tensor(str(tmp_path), "blk.1.ffn_down.weight")
    assert dt == "q4_0" and shape == (256, 704) and raw.size == 256 * 704 // 32 * 18
    import numpy as np
    from gguf import GGMLQuantizationType as T
    from gguf import quants

    w = quants.dequantize(raw.reshape(256, -1), T.Q4_0)
    assert np.isfinite(w).all() and 0.005 < float(w.std()) < 0.05
