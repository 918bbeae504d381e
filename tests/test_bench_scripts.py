"""benchmark/bench_configs.py dry run on CPU/gloo (``--tiny``): the script that reports the BASELINE.json configs and
their roofline fractions keeps working without a GPU in the loop."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_configs_tiny_world2():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", "29691", os.path.join(ROOT, "benchmark", "bench_configs.py"), "--tiny"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:]
    rows = [json.loads(line) for line in r.stdout.splitlines() if line.startswith("{")]
    assert [x["config"] for x in rows] == ["zigzag", "varlen", "llama3", "stripe8"]
    for x in rows:
        assert x["n_gpus"] == 2 and x["ms_per_step"] > 0
        roof = x["roofline"]
        assert roof["compute_ms"] > 0 and roof["nvlink_ms"] > 0 and roof["bound"] in ("compute", "nvlink")


def test_bench_reference_arm_reports_unavailable_without_a_gpu():
    """The driver contract: `bench.py --impl reference` prints one JSON line and exits 0 when it cannot run."""
    import torch

    if torch.cuda.is_available():
        import pytest

        pytest.skip("CPU-only check")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference"], stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-1000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and "unavailable" in line
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                       text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0 and "CUDA" in (r.stderr + r.stdout)


def test_prefetched_e2e_loop_pipelines_one_copy_per_step():
    """bench.PrefetchedE2E with synchronous stand-ins for torch.cuda: step i must consume exactly the inputs that
    were on the host when step i-1 ran (copied while step i-1 'computed'), from alternating buffers, one host->device
    copy per step."""
    import contextlib
    import importlib.util

    import torch

    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)

    log = []

    class Event:
        def record(self, stream=None):
            log.append("record")

    class Stream:
        def __init__(self, device=None):
            pass

        def wait_event(self, ev):
            pass

        def synchronize(self):
            pass

    _Event, _Stream = Event, Stream

    class Cuda:
        Event, Stream = _Event, _Stream

        @staticmethod
        @contextlib.contextmanager
        def stream(s):
            yield

        @staticmethod
        def current_stream():
            return Stream()

    host = [torch.zeros(4)]
    seen = []

    def step(ins):
        seen.append((float(ins[0][0]), ins[0].data_ptr()))
        return ins[0] * 1.0

    loss_host = torch.zeros(1)
    e2e = bench.PrefetchedE2E(Cuda, torch, torch.device("cpu"), host, step, loss_host, False)
    for i in range(5):
        host[0].fill_(float(i + 1))  # what the "data loader" holds while step i runs = inputs of step i+1
        loss = e2e()
        assert loss == float(i)  # step i sees the value the host held one call earlier (0 at construction)
    assert [v for v, _ in seen] == [0.0, 1.0, 2.0, 3.0, 4.0]
    ptrs = [p for _, p in seen]
    assert ptrs[0] == ptrs[2] == ptrs[4] and ptrs[1] == ptrs[3] and ptrs[0] != ptrs[1]  # double buffer alternates


def test_dump_sample_is_fixed_float32_and_small():
    """bench.sample_rows (what ``--dump-outputs`` writes): the same token rows of every array on every run, exact
    float32 copies of the bf16 values, and at most 64 MB at the headline shape whatever the GPU count."""
    import importlib.util

    import torch

    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)

    tokens = 2048
    pos = torch.arange(tokens, dtype=torch.float32).view(1, tokens, 1, 1).expand(1, tokens, 2, 4).contiguous()
    arrays = {"out": pos, "dqkv": torch.randn(1, tokens, 3, 2, 4, dtype=torch.bfloat16).requires_grad_(True)}
    a, b = bench.sample_rows(torch, arrays, 1), bench.sample_rows(torch, arrays, 1)
    rows = a["out"][0, :, 0, 0].astype(int)
    assert a.keys() == arrays.keys() and all(x.dtype.name == "float32" for x in a.values())
    assert a["out"].shape == (1, bench.DUMP_ROWS, 2, 4) and a["dqkv"].shape == (1, bench.DUMP_ROWS, 3, 2, 4)
    assert all((a[k] == b[k]).all() for k in a)  # same rows every run
    assert (rows[1:] > rows[:-1]).all()
    assert (a["dqkv"] == arrays["dqkv"].detach()[:, rows].float().numpy()).all()  # same rows, exact values
    assert bench.sample_rows(torch, arrays, 8)["out"].shape[1] == bench.DUMP_ROWS // 8
    per_row = 32 * 128 * 4 * (1 + 3)  # out + dqkv of one headline token row, float32
    assert bench.DUMP_ROWS * per_row <= 64 * 2**20


def test_minimal_example_world2():
    """examples/ring_attention_minimal.py: shard, attend, backward, sampled fp32 check - on gloo."""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", "29693", os.path.join(ROOT, "examples", "ring_attention_minimal.py"),
           "--scheme", "stripe", "--head-dim", "64"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0 and "ok=True" in r.stdout, r.stdout[-2000:]
