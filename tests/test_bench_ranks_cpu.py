"""N > 1 path of bench.py on CPU: world_size-2 gloo run of the rank aggregation (replicas only: MAX of times, SUM of work)."""
import os
import sys

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    import bench

    dist.init_process_group("gloo", rank=rank, world_size=world)
    # rank r: device leg took 100 + 50 r ms for 10 + r audio seconds, e2e leg 200 - 20 r ms for 5 audio seconds
    times, totals = bench.aggregate_over_ranks([100.0 + 50.0 * rank, 200.0 - 20.0 * rank], [10.0 + rank, 5.0], "cpu", world)
    out[rank] = (times, totals)
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_aggregation_over_gloo():
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    port = 29500 + (os.getpid() % 2000)
    mp.spawn(_worker, args=(world, port, out), nprocs=world, join=True)
    for r in range(world):
        times, totals = out[r]
        assert times == [150.0, 200.0]          # max over ranks, per leg
        assert totals == [21.0, 10.0]           # whole-job audio seconds
    # value = whole-job audio seconds / max time, as bench.py reports it
    assert abs(out[0][1][0] / (out[0][0][0] * 1e-3) - 140.0) < 1e-9


def test_single_rank_is_identity():
    sys.path.insert(0, ROOT)
    import bench

    times, totals = bench.aggregate_over_ranks([12.5], [3.0], "cpu", 1)
    assert times == [12.5] and totals == [3.0]


def test_reference_arm_prints_the_contract_line_on_rank_0_only():
    """`bench.py --impl reference` (the CPU arm): rank 0 prints ONE JSON line with the contract's keys, the same metric / unit /
    config keys as the B200 arm, a cpu_baseline describing this run and an e2e equal to the line's value; other ranks exit 0
    without work.  Tiny preset, one 8-frame step: the arm's code path, not its number."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--model", "tiny-Base", "--steps", "1", "--warmup", "0",
           "--cpu-frames", "8", "--gpus", "2"]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    r0 = subprocess.run(cmd, env=dict(env, RANK="0", WORLD_SIZE="2"), capture_output=True, text=True, timeout=300)
    assert r0.returncode == 0, r0.stderr[-2000:]
    lines = [l for l in r0.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e", "impl"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "audio_seconds_per_second" and d["unit"] == "audio-s/s" and d["n_gpus"] == 2
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1
    assert "workload" in d["config"] and "model" not in d["config"] and d["config"]["reference_sample"]["frames_per_step"] == 8
    r1 = subprocess.run(cmd, env=dict(env, RANK="1", WORLD_SIZE="2"), capture_output=True, text=True, timeout=300)
    assert r1.returncode == 0 and r1.stdout.strip() == ""


def test_zero_steps_and_a_dump_from_the_cpu_arm_are_refused(tmp_path):
    """--steps sets the number of timed steps, so fewer than one is an error; --dump-outputs writes the B200 arm's outputs and is
    refused for the CPU arm instead of being ignored.  Nothing is written."""
    import subprocess

    bench = os.path.join(ROOT, "bench.py")
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "d")]):
        r = subprocess.run([sys.executable, bench] + args, capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and "error" in r.stderr, (args, r.stderr[-500:])
    assert not (tmp_path / "d").exists()
