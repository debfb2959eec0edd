"""bench.py's supervisor (CPU self-test mode, canned numbers): the measurement and the same-box baselines run as child
processes with their own rendezvous port / job id and WITHOUT torchrun's agent-store variables; a configuration that
fails or hangs on some rank is replaced by the conservative one on every rank; a failing baseline arm costs only its
own entry; rank 0 prints exactly one JSON line."""
import json
import os
import subprocess
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _launch(world, selftest, port, arm_timeout=6, attempt_timeout=20, extra=""):
    """All ranks share one parent (like torchrun's agent): a small shell that backgrounds ranks 1.. and runs rank 0."""
    lines = []
    for r in range(world - 1, -1, -1):
        cmd = (f"RANK={r} LOCAL_RANK={r} WORLD_SIZE={world} MASTER_ADDR=127.0.0.1 MASTER_PORT={port} TORCHELASTIC_USE_AGENT_STORE=True "
               f"TORCHELASTIC_RUN_ID=none B200MPI_BENCH_SELFTEST={selftest} {sys.executable} {REPO}/bench.py --gpus {world} --steps 3 "
               f"--warmup 3 --arm-timeout {arm_timeout} --attempt-timeout {attempt_timeout} {extra}")
        lines.append(cmd + (" > /dev/null 2>&1 &" if r else ""))
    lines.append("rc=$?; wait; exit $rc")
    return subprocess.run(["sh", "-c", "\n".join(lines)], capture_output=True, text=True, timeout=240)


@pytest.mark.parametrize("world", [1, 2])
def test_one_line_with_same_box_ratios_and_clean_child_env(world):
    r = _launch(world, "ok", 29810 + world)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["value"] == 4000.0 * world and d["config"]["bench_configuration"] == "default"
    assert d["config"]["agent_store"] is None            # torchrun's store settings must not leak into the children
    assert d["config"]["port"] != str(29810 + world)     # own rendezvous port
    sb = d["same_box"]
    assert sb["ratio_vs_nccl"] == pytest.approx(4000 / 3900, abs=1e-3) and sb["ratio_vs_torchddp"] == 2.0
    assert sb["nccl_same_engine"]["impl"] == "nccl" and sb["torchddp_stock"]["impl"] == "torchddp"


def test_faster_multi_gpu_candidate_is_the_one_reported():
    """world > 1: the default configuration and the one with the bf16 shadow + small tail bucket are both measured in full;
    the line carries the faster one and lists both."""
    r = _launch(2, "full_faster", 29825)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["config"]["bench_configuration"] == "full" and d["value"] == pytest.approx(8400.0)
    assert set(d["config"]["candidates"]) == {"default", "full"}
    assert d["same_box"]["ratio_vs_nccl"] == pytest.approx(8400 / 7800, abs=1e-3)


def test_dump_outputs_are_those_of_the_reported_candidate(tmp_path):
    """--dump-outputs DIR: every candidate dumps, DIR receives the files of the one the line reports and nothing else."""
    import numpy as np
    out = tmp_path / "out"
    r = _launch(2, "full_faster", 29826, extra=f"--dump-outputs {out}")
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][0])
    assert d["config"]["bench_configuration"] == "full"
    assert sorted(os.listdir(out)) == ["buffers.npy", "loss.npy", "params.npy"]
    assert float(np.load(out / "loss.npy")) == pytest.approx(d["value"])
    assert np.load(out / "params.npy").dtype == np.float32


def test_dump_outputs_samples_large_parameter_sets_the_same_way_every_time(tmp_path):
    import numpy as np
    import torch
    import bench
    n = bench.DUMP_SAMPLE + 12344
    params = [torch.arange(n, dtype=torch.float32).reshape(-1, 4)]
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), torch.tensor(1.5), params, [torch.ones(4), torch.zeros(2, dtype=torch.long)])
    a, b = np.load(tmp_path / "a" / "params.npy"), np.load(tmp_path / "b" / "params.npy")
    assert a.dtype == np.float32 and a.shape == (bench.DUMP_SAMPLE,) and np.array_equal(a, b)
    assert (np.diff(a) > 0).all() and a[-1] < n               # distinct positions, in order (each value is its position)
    assert np.load(tmp_path / "a" / "buffers.npy").tolist() == [1.0] * 4      # integer buffers are left out
    assert float(np.load(tmp_path / "a" / "loss.npy")) == 1.5


def test_failing_default_configuration_falls_back_on_every_rank():
    r = _launch(2, "fail_default", 29821)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][0])
    assert d["config"]["bench_configuration"] == "conservative" and d["value"] == 8000.0
    assert any("default" in n for n in d["config"]["earlier_attempts"])


def test_hang_on_one_rank_is_cut_off_and_replaced():
    r = _launch(2, "hang_default", 29822, attempt_timeout=5)
    # the hanging rank is rank 1; rank 0's child succeeds, the agreement fails after rank 1's child is killed
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][0])
    assert d["config"]["bench_configuration"] == "conservative"


def test_failing_baseline_arm_is_reported_not_fatal():
    r = _launch(1, "fail_nccl", 29823)
    assert r.returncode == 0
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][0])
    assert "error" in d["same_box"]["nccl_same_engine"] and d["same_box"]["ratio_vs_nccl"] is None
    assert d["same_box"]["ratio_vs_torchddp"] == 2.0


def test_arms_are_skipped_when_the_time_budget_is_spent():
    env = dict(os.environ, B200MPI_BENCH_SELFTEST="ok", B200MPI_BENCH_BUDGET_S="30", MASTER_PORT="29824")
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        env.pop(k, None)
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--steps", "3", "--warmup", "3"], capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][0])
    assert d["value"] == 4000.0 and "skipped" in d["same_box"]["nccl_same_engine"] and d["same_box"]["ratio_vs_nccl"] is None
