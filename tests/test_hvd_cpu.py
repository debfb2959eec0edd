"""CPU-checkable parts of the Horovod-compatible front-end: Adasum math, elastic State bookkeeping, API surface."""
import os

import pytest
import torch

import horovod.torch as hvd
from mpi_operator_b200.hvd.adasum import adasum_pair, adasum_tree


def test_adasum_properties():
    a = torch.tensor([1.0, 0.0, 0.0])
    b = torch.tensor([0.0, 2.0, 0.0])
    torch.testing.assert_close(adasum_pair(a, b), a + b)          # orthogonal gradients add
    torch.testing.assert_close(adasum_pair(a, a), a)              # identical gradients average
    torch.testing.assert_close(adasum_pair(a, 3 * a), 2.0 * a)    # parallel gradients: (a + 3a)/2
    z = torch.zeros(3)
    torch.testing.assert_close(adasum_pair(a, z), a)              # zero gradient is neutral
    ts = [torch.randn(50) for _ in range(5)]                      # non power-of-two tree is well defined
    out = adasum_tree(ts)
    assert out.shape == (50,) and torch.isfinite(out).all()
    torch.testing.assert_close(adasum_tree([ts[0]]), ts[0])
    torch.testing.assert_close(adasum_tree(ts[:2]), adasum_pair(ts[0], ts[1]))


def test_hvd_surface_and_uninitialised_errors():
    for name in ("init", "shutdown", "rank", "size", "local_rank", "local_size", "allreduce", "allreduce_", "allgather", "broadcast",
                 "broadcast_", "broadcast_parameters", "broadcast_optimizer_state", "broadcast_object", "DistributedOptimizer",
                 "Average", "Sum", "Adasum", "Compression", "elastic", "nccl_built", "mpi_built", "join", "barrier"):
        assert hasattr(hvd, name), name
    assert hvd.nccl_built() and hvd.Average == "average"
    if not hvd.is_initialized():
        with pytest.raises(RuntimeError):
            hvd.rank()


def test_elastic_state_commit_restore_and_host_update(tmp_path, monkeypatch):
    from mpi_operator_b200.hvd import elastic
    root = tmp_path / "rootfs"
    (root / "etc/mpi").mkdir(parents=True)
    script = root / "etc/mpi/discover_hosts.sh"
    script.write_text("#!/bin/sh\necho a\n")
    monkeypatch.setenv("B200MPI_POD_ROOTFS", str(root))
    st = elastic.State(step=0, note="x")
    st.step = 7
    st.commit()                       # saves, host set unchanged
    st.step = 9
    st.restore()
    assert st.step == 7
    script.write_text("#!/bin/sh\necho a\necho b\n")
    st.step = 8
    with pytest.raises(elastic.HostsUpdatedInterrupt):
        st.commit()                   # saved first, then the changed host set interrupts
    st.step = 100
    st.restore()
    assert st.step == 8

    resets = []
    st.register_reset_callbacks([lambda: resets.append(st.step)])
    assert elastic.ObjectState is elastic.State

    @elastic.run
    def train(state):
        assert resets == [8]          # on_reset ran after restore + sync, before the training function
        raise elastic.HostsUpdatedInterrupt("rescale")
    monkeypatch.setattr(elastic.State, "sync", lambda self: None)
    with pytest.raises(SystemExit) as e:
        train(st)
    assert e.value.code == 75

    @elastic.run
    def broken(state):       # a dead peer / shut-down engine surfaces as HorovodInternalError: roll back, leave for a re-spawn
        state.step = 12345
        raise hvd.HorovodInternalError("rank 1 died", -5)
    st.step = 8
    st.save()
    with pytest.raises(SystemExit) as e:
        broken(st)
    assert e.value.code == 75 and st.step == 8


def test_trace_export_and_roofline_report(tmp_path):
    import json
    from mpi_operator_b200.utils import roofline, trace
    p = tmp_path / "t.jsonl"
    p.write_text("\n".join(json.dumps(r) for r in [
        {"rank": 0, "op": "allreduce", "bytes": 1024, "algo": "oneshot", "blocks": 1, "t_ns": 1000},
        {"rank": 1, "op": "allreduce", "bytes": 1024, "algo": "oneshot", "blocks": 1, "t_ns": 1500},
        {"rank": 0, "op": "allreduce_sgd", "bytes": 1 << 25, "algo": "nvls", "blocks": 16, "t_ns": 9000}]))
    out = tmp_path / "t.json"
    assert trace.main([str(p), str(out)]) == 0
    ev = json.load(open(out))["traceEvents"]
    assert sum(1 for e in ev if e["ph"] == "X") == 3 and {e["pid"] for e in ev} == {0, 1}
    assert trace.summarize(trace.load_jsonl(str(p)))["allreduce[oneshot]"] == {"calls": 2, "bytes": 2048}
    md = roofline.report(os.path.join(_repo(), "profiles", "allreduce_sweep_n8_f32.json"))
    assert "| float32 | 1073741824 | nvls" in md and "x |" in md


def _repo():
    import os as _os
    return _os.path.dirname(_os.path.dirname(_os.path.abspath(__file__)))


@pytest.mark.parametrize("np_,engine", [(1, "1"), (4, "1"), (3, "0")])
def test_horovod_api_on_the_cpu_backend_under_mpirun(np_, engine):
    """The reference's Horovod example is a CPU job (examples/v2beta1/horovod/tensorflow-mnist.yaml: cpu-only workers).
    Without CUDA, hvd.init() builds the libmpi-shim communicator (hvd/host_backend.py); tests/hvd_cpu_worker.py checks
    every collective, DistributedOptimizer against SGD on the averaged gradient, Adasum and the elastic State."""
    import os
    import subprocess
    import sys
    repo = _repo()
    mpirun = os.path.join(repo, "mpi_operator_b200/bin/mpirun")
    if not os.path.exists(mpirun):
        pytest.skip("native launcher not built (run make)")
    env = dict(os.environ, B200MPI_HVD_DEVICE="cpu", B200MPI_HVD_ENGINE=engine)   # "0": direct call-order path over the libmpi shim
    r = subprocess.run([mpirun, "-np", str(np_), sys.executable, os.path.join(repo, "tests/hvd_cpu_worker.py")],
                       capture_output=True, text=True, timeout=180, env=env, cwd="/tmp")
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert r.stdout.count("hvd cpu ok") == np_


def test_affinity_helper_is_a_safe_no_op_without_nvml(monkeypatch):
    from mpi_operator_b200.utils import affinity
    before = os.sched_getaffinity(0)
    assert affinity.bind_to_gpu(0) is None or affinity.bind_to_gpu(0) <= before
    monkeypatch.setenv("B200MPI_NO_AFFINITY", "1")
    assert affinity.bind_to_gpu(0) is None
    monkeypatch.delenv("B200MPI_NO_AFFINITY")
    monkeypatch.setattr(affinity, "gpu_cpu_set", lambda i: {min(before)})     # a GPU-local set inside the allowed set
    got = affinity.bind_to_gpu(0)
    try:
        assert (got == {min(before)} and os.sched_getaffinity(0) == {min(before)}) or len(before) == 1
        monkeypatch.setattr(affinity, "gpu_cpu_set", lambda i: {10 ** 6})     # disjoint from what the cgroup allows
        assert affinity.bind_to_gpu(0) is None
    finally:
        os.sched_setaffinity(0, before)


def test_horovod_package_layout_and_programmatic_run():
    """Deep imports scripts use (`horovod.torch.elastic`, `horovod.torch.mpi_ops`, `horovod.common.exceptions`, ...) and
    `horovod.run(fn, np=N)`: the function runs on N ranks under the native mpirun, results come back in rank order."""
    import horovod
    import horovod.torch.elastic as hvde
    from horovod.common.exceptions import HorovodInternalError, HostsUpdatedInterrupt
    from horovod.common.util import mpi_built, nccl_built
    from horovod.torch.compression import Compression
    from horovod.torch.functions import broadcast_parameters
    from horovod.torch.mpi_ops import allreduce_async_, poll, synchronize
    from horovod.torch.optimizer import DistributedOptimizer
    from horovod.torch.sync_batch_norm import SyncBatchNorm
    assert HorovodInternalError is hvd.HorovodInternalError and HostsUpdatedInterrupt is hvde.HostsUpdatedInterrupt
    assert hvde.run is hvd.elastic.run and Compression is hvd.Compression and SyncBatchNorm is hvd.SyncBatchNorm
    assert callable(allreduce_async_) and callable(poll) and callable(synchronize) and callable(broadcast_parameters)
    assert DistributedOptimizer is hvd.DistributedOptimizer and mpi_built() and nccl_built()
    if not os.path.exists(os.path.join(_repo(), "mpi_operator_b200/bin/mpirun")):
        pytest.skip("native launcher not built (run make)")

    def sum_of_ranks(offset):
        import torch as t
        import horovod.torch as h
        h.init()
        out = float(h.allreduce(t.tensor([float(h.rank() + offset)]), op=h.Sum))
        r = h.rank()
        h.shutdown()
        return r, out
    res = horovod.run(sum_of_ranks, args=(10,), np=3, env={"B200MPI_HVD_DEVICE": "cpu"})
    assert res == [(0, 33.0), (1, 33.0), (2, 33.0)]


def test_mnist_example_with_the_use_adasum_flag():
    """The reference example's optional ``--use-adasum`` (tensorflow_mnist.py:31-32,126-133): DistributedOptimizer(op=Adasum)
    combines the ranks' model deltas; on host tensors through the native engine (hvd_core.cc host_adasum)."""
    import os
    import re
    import subprocess
    import sys
    repo = _repo()
    mpirun = os.path.join(repo, "mpi_operator_b200/bin/mpirun")
    if not os.path.exists(mpirun):
        pytest.skip("native launcher not built (run make)")
    env = dict(os.environ, B200MPI_HVD_DEVICE="cpu")
    r = subprocess.run([mpirun, "-np", "2", sys.executable, os.path.join(repo, "examples/horovod/torch_mnist.py"), "--use-adasum",
                        "--steps", "60"], capture_output=True, text=True, timeout=240, env=env, cwd="/tmp")
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    losses = [float(x) for x in re.findall(r"loss = ([0-9.]+)", r.stdout)]
    assert len(losses) >= 3 and losses[-1] < 0.25 * losses[0], losses


def test_tf_cnn_benchmarks_train_dir_checkpoints_and_resumes(tmp_path):
    """tf_cnn_benchmarks' --train_dir: rank 0 writes a checkpoint at the end, the next run restores it on every rank
    (SURVEY.md section 5.4; rank-0-only writer as in the reference's tensorflow_mnist.py:159)."""
    import os
    import subprocess
    import sys
    repo = _repo()
    mpirun = os.path.join(repo, "mpi_operator_b200/bin/mpirun")
    if not os.path.exists(mpirun):
        pytest.skip("native launcher not built (run make)")
    script = os.path.join(repo, "examples/tensorflow-benchmarks/scripts/tf_cnn_benchmarks/tf_cnn_benchmarks.py")
    cmd = [mpirun, "-np", "2", sys.executable, script, "--device=cpu", "--model=trivial", "--batch_size=4", "--num_batches=3",
           "--num_warmup_batches=1", "--image_size=32", "--train_dir", str(tmp_path / "ckpt")]
    env = dict(os.environ, B200MPI_HVD_DEVICE="cpu")
    first = subprocess.run(cmd, capture_output=True, text=True, timeout=240, env=env, cwd="/tmp")
    assert first.returncode == 0 and "Saved checkpoint" in first.stdout and "Restored" not in first.stdout, first.stdout[-1500:] + first.stderr[-2000:]
    second = subprocess.run(cmd, capture_output=True, text=True, timeout=240, env=env, cwd="/tmp")
    assert second.returncode == 0 and "Restored checkpoint" in second.stdout and "written after 4 batches on 2 ranks" in second.stdout, \
        second.stdout[-1500:] + second.stderr[-2000:]
    # --eval=True: forward only through DataParallelTrainer.evaluate, restoring the checkpoint the OTHER engine wrote
    third = subprocess.run(cmd + ["--eval=True"], capture_output=True, text=True, timeout=240, env=env, cwd="/tmp")
    assert third.returncode == 0 and "Restored checkpoint" in third.stdout and "Saved checkpoint" not in third.stdout, third.stdout[-1500:] + third.stderr[-2000:]
    import re
    m = re.search(r"Accuracy @ 1 = ([0-9.]+) Accuracy @ 5 = ([0-9.]+) \[(\d+) examples\]", third.stdout)
    assert m and 0.0 <= float(m.group(1)) <= float(m.group(2)) <= 1.0 and int(m.group(3)) == 3 * 4 * 2


def _adasum_kernel_model(vectors, ctas=3):
    """Host model of csrc/kernels/adasum.cu (same index arithmetic, one Python loop per CTA): rank r owns slice r of every
    vector in its work area W; per level every (rank, CTA) publishes 3 partial sums per pair in its own board slot, the board
    is summed over (rank, CTA), the slice is combined in place at W[g] with g = p * 2 * dist, h = g + dist, and the partial
    dots of the NEXT level are accumulated in the same pass (even pair -> `prev`, odd pair -> dot with `prev`); the last level
    writes the slice to every rank's A. Returns every rank's A."""
    import torch
    world, n = len(vectors), vectors[0].numel()
    per = -(-n // world)
    pad = [torch.cat([v.double(), torch.zeros(world * per - n, dtype=torch.float64)]) for v in vectors]
    A = [torch.stack(pad).clone() for _ in range(world)]                       # A[rank][q] = rank's copy of vector q (phase 0 + barrier)
    W = [torch.stack([pad[q][r * per:(r + 1) * per] for q in range(world)]) for r in range(world)]   # level-0 pull: slice r of all q
    chunks = [list(torch.arange(per).chunk(ctas)) for _ in range(world)]
    # partial dots of the level-0 pairs (2p, 2p+1), per (rank, cta)
    np_ = world // 2
    acc = {(r, c): [(float(W[r][2 * p][idx] @ W[r][2 * p + 1][idx]), float(W[r][2 * p][idx] @ W[r][2 * p][idx]),
                     float(W[r][2 * p + 1][idx] @ W[r][2 * p + 1][idx])) for p in range(np_)]
           for r in range(world) for c, idx in enumerate(chunks[r])}
    board, pair_base, dist = {}, 0, 1
    while dist < world:
        for (r, c), sums in acc.items():
            for p, s in enumerate(sums):
                board[(pair_base + p, r, c)] = s                               # own slot: nothing to zero between levels
        coef = []
        for p in range(np_):
            d, na, nb = (sum(board[(pair_base + p, r, c)][k] for r in range(world) for c in range(len(chunks[r]))) for k in range(3))
            coef.append((1.0 - d / (2 * na) if na > 0 else 1.0, 1.0 - d / (2 * nb) if nb > 0 else 1.0))
        last = np_ == 1
        nxt = {}
        for r in range(world):
            for c, idx in enumerate(chunks[r]):
                sums, prev = [], None
                for p in range(np_):
                    g, h = p * 2 * dist, p * 2 * dist + dist
                    z = coef[p][0] * W[r][g][idx] + coef[p][1] * W[r][h][idx]
                    if last:
                        for q in range(world):
                            A[q][0][r * per + idx] = z                           # slice push: the all-gather half (result lives in row 0 here)
                    else:
                        W[r][g][idx] = z
                        if p & 1:
                            sums.append((float(prev @ z), float(prev @ prev), float(z @ z)))
                        else:
                            prev = z
                nxt[(r, c)] = sums
        acc, pair_base, np_, dist = nxt, pair_base + np_, np_ // 2, dist * 2
    return [a[0][:n] for a in A]


def test_adasum_kernel_index_model_matches_tree():
    """The slice-parallel, level-fused schedule of the device kernel reproduces the pairwise tree (any size, 2/4/8 ranks,
    more CTAs than elements, zero vectors) - checks the pair / slot / next-level-dot index arithmetic without a GPU."""
    import torch
    g = torch.Generator().manual_seed(0)
    for world in (2, 4, 8):
        for n in (1, 5, 64, 257):
            vs = [torch.randn(n, generator=g, dtype=torch.float64) * (1 + r) for r in range(world)]
            if n == 64:
                vs[1].zero_()
            want = adasum_tree(vs)
            for ctas in (1, 3):
                outs = _adasum_kernel_model(vs, ctas=ctas)
                for o in outs:
                    assert torch.allclose(o, want, rtol=1e-12, atol=1e-12), (world, n, ctas)
