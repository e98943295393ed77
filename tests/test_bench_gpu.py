"""bench.py --dump-outputs on the GPU, tiny preset: the last timed step's codes and audio land in DIR as float32 .npy, and two runs
with the same arguments write the same arrays (seeded sampling), so two builds of the project can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--model", "tiny-Base", "--frames", "24", "--chunk", "8", "--steps", "2",
           "--warmup", "3", "--batched-streams", "0", "--serving-requests", "0", "--anchor-frames", "0", "--no-cpu-baseline",
           "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=500)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_dump_outputs_hold_the_last_timed_step_and_repeat(tmp_path):
    from qwen3_tts_cuda_graphs_b200.config import preset

    cfg = preset("tiny-Base")
    assert _bench(tmp_path / "a")["steps"] == 2
    assert sorted(os.listdir(tmp_path / "a")) == ["audio.npy", "codes.npy"]
    codes, audio = np.load(tmp_path / "a" / "codes.npy"), np.load(tmp_path / "a" / "audio.npy")
    assert codes.dtype == np.float32 and codes.shape == (24, cfg.talker.num_code_groups)
    assert np.array_equal(codes, np.round(codes)) and codes.min() >= 0
    # one utterance of 24 frames: every chunk of it decoded, nothing of another step
    assert audio.dtype == np.float32 and audio.shape == (cfg.codec.n_samples(24),) and np.isfinite(audio).all()
    _bench(tmp_path / "b")
    assert np.array_equal(np.load(tmp_path / "b" / "codes.npy"), codes)
    assert np.array_equal(np.load(tmp_path / "b" / "audio.npy"), audio)
