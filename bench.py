#!/usr/bin/env python
"""Headline benchmark: zigzag ring flash attention, fwd+bwd iterations per second.

Config (BASELINE.json "headline"): ``zigzag_ring_flash_attn_qkvpacked_func``, bf16, batch 1, sequence 32768,
32 heads, head_dim 128, causal, synthetic random Q/K/V.  The sequence is fixed and sharded over the N GPUs
(strong scaling: 32768/N tokens per GPU, total attention work constant).  One step = forward + backward of
the attention op through the public API.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--config readme]

``--impl reference`` runs the unmodified zhuzilin/ring-flash-attention installed in ``baseline/_ref``
(flash_attn 2.8 + NCCL) on the same config and prints the same JSON line with ``"impl": "reference"``.
``--config readme`` switches to the reference README's benchmark shape (8192 tokens per GPU, 32 query / 8 kv
heads, kvpacked API), for which published H800 numbers exist (BASELINE.md).

Timing: CUDA events around every step on the launching stream, an L2 flush (256 MiB write) between steps,
barrier + synchronize on both sides of the timed region, max over ranks.  ``e2e`` repeats the measurement
with the step's inputs copied from pinned host memory and the loss read back every step; the copy of step i+1 is
prefetched on a side stream into a double buffer while step i computes (same loop for both arms,
``RFA_BENCH_E2E_PREFETCH=0`` serialises copy and compute again).

``--dump-outputs DIR`` writes what the last timed step returned to its caller (the attention output and, for
fwd_bwd, the gradients of the inputs) as float32 ``DIR/<name>.npy``, each cut down to the same fixed, seeded
sample of token rows (``_rank<r>`` is appended to the name when N > 1).  Inputs are seeded too, so two builds run
with the same arguments can be compared array for array.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading

ROOT = os.path.dirname(os.path.abspath(__file__))

PUBLISHED = {  # BASELINE.md, README config, fwd+bwd iter/s
    ("readme", 8): 17.4,   # zigzag_ring, 8xH800
    ("readme", 1): 154.7,  # flash_attn on the local 8K problem, 1xH800 (zigzag at world 1 is exactly this)
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="headline", choices=["headline", "readme"])
    ap.add_argument("--mode", default="fwd_bwd", choices=["fwd_bwd", "fwd"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--check", dest="check", action="store_true", default=True,
                    help="verify one untimed step against the fp32 oracle on sampled rows (default: on, ours only)")
    ap.add_argument("--no-check", dest="check", action="store_false")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed sample of the last timed step's outputs as float32 DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_ROWS = 512  # token rows dumped over all ranks: 32 MiB of float32 at the headline shape


def sample_rows(torch, arrays, world):
    """The same seeded sample of token rows (dim 1) of every array, as float32 numpy arrays."""
    n = next(iter(arrays.values())).shape[1]
    rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[: max(1, DUMP_ROWS // world)].sort().values
    return {name: t.detach()[:, rows.to(t.device)].float().cpu().numpy() for name, t in arrays.items()}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except ValueError:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7),
                              ("sw_power_cap", 8)):
                if r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def unavailable(why: str):
    print(json.dumps({"impl": "reference", "unavailable": why}))
    sys.exit(0)


def load_reference():
    """Import the UNMODIFIED reference from baseline/_ref.  Its package __init__ eagerly imports the HF
    adapter, which does not import under transformers 5.x; a stub module object for that one submodule is
    registered first so that the algorithm modules (the code path being benchmarked) load untouched."""
    ref_root = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_root, "ring_flash_attn")):
        unavailable("baseline/_ref/ring_flash_attn is not installed")
    try:
        import flash_attn  # noqa: F401
    except Exception as e:  # noqa: BLE001
        unavailable(f"flash_attn import failed: {type(e).__name__}: {e}")
    sys.path.insert(0, ref_root)
    import types

    stub = types.ModuleType("ring_flash_attn.adapters")
    stub.substitute_hf_flash_attn = None
    stub.update_ring_flash_attn_params = None
    sys.modules["ring_flash_attn.adapters"] = stub
    try:
        import ring_flash_attn
    except Exception as e:  # noqa: BLE001
        unavailable(f"reference import failed: {type(e).__name__}: {e}")
    if not os.path.abspath(ring_flash_attn.__file__).startswith(os.path.abspath(ref_root)):
        unavailable("ring_flash_attn resolved outside baseline/_ref")
    return ring_flash_attn


class PrefetchedE2E:
    """The end-to-end step with the input pipeline every training loop has: while step i computes, the host->device
    copy of step i+1's inputs (from the same pinned host tensors) runs on a side stream into the other half of a
    double buffer.  Every step's inputs are still copied from pinned host memory inside the timed region (one copy
    per timed step) and the loss is read back every step; only the serialisation of copy and compute is gone.
    Used for both arms (RFA_BENCH_E2E_PREFETCH=0 restores the serial loop).

    ``cuda`` is ``torch.cuda`` (a stand-in with the same five names in tests/test_bench_scripts.py)."""

    def __init__(self, cuda, torch, dev, host_in, step, loss_host, needs_grad):
        self.cuda, self.step, self.host_in, self.loss_host, self.needs_grad = cuda, step, host_in, loss_host, needs_grad
        self.copy_stream = cuda.Stream(device=dev)
        self.bufs = [[torch.empty(h.shape, dtype=h.dtype, device=dev) for h in host_in] for _ in range(2)]
        self.ready = [cuda.Event(), cuda.Event()]
        self.consumed = [cuda.Event(), cuda.Event()]
        self.i = 0
        self._prefetch(0)

    def _prefetch(self, i):
        b = i & 1
        with self.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self.consumed[b])  # the step that last read this half has finished
            for d, h in zip(self.bufs[b], self.host_in):
                d.copy_(h, non_blocking=True)
            self.ready[b].record(self.copy_stream)

    def __call__(self):
        i, b = self.i, self.i & 1
        self.i += 1
        self._prefetch(i + 1)  # next step's inputs travel while this step computes
        cur = self.cuda.current_stream()
        cur.wait_event(self.ready[b])
        ins = [d.detach().requires_grad_(self.needs_grad) for d in self.bufs[b]]
        out = self.step(ins)
        self.loss_host.copy_(out.float().mean().reshape(1), non_blocking=True)
        self.consumed[b].record(cur)
        cur.synchronize()
        return float(self.loss_host[0])


def run_check(torch, fn, api, dev_in, dout, group):
    """One untimed fwd+bwd through the public API at the benchmark shape and world size, compared on sampled rows
    with an fp32 oracle built from all-gathered inputs (ring_flash_attn_b200/utils/verify.py)."""
    from ring_flash_attn_b200.utils.verify import sampled_check

    for t in dev_in:
        t.grad = None
    out, lse, _ = fn(*dev_in, causal=True, return_attn_probs=True)
    out.backward(dout)
    if api == "qkvpacked":
        qkv, g = dev_in[0].detach()[0], dev_in[0].grad[0]
        q, k, v, dq, dk, dv = qkv[:, 0], qkv[:, 1], qkv[:, 2], g[:, 0], g[:, 1], g[:, 2]
    else:
        q, kv = dev_in[0].detach()[0], dev_in[1].detach()[0]
        k, v, dq = kv[:, 0], kv[:, 1], dev_in[0].grad[0]
        dk, dv = dev_in[1].grad[0][:, 0], dev_in[1].grad[0][:, 1]
    res = sampled_check("zigzag", q, k, v, dout[0], out.detach()[0], lse[0], dq, dk, dv, group=group)
    for t in dev_in:
        t.grad = None
    return {"ok": res["ok"], "max_err": res["max_err"], "tol": res["tol"], "rows": res["rows"],
            "heads": res["heads_q"], "what": "sampled rows vs fp32 oracle from all-gathered inputs"}


def main():
    args = parse()
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        if args.impl == "reference":
            unavailable("no CUDA device")
        raise SystemExit("bench.py needs a CUDA device")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    need_pg = world > 1 or args.impl == "reference"
    if need_pg and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29513")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    if args.config == "headline":
        tokens, hq, hkv, api, scaling = 32768 // world, 32, 32, "qkvpacked", "strong"
    else:
        tokens, hq, hkv, api, scaling = 8192, 32, 8, "kvpacked", "weak"
    d = 128
    dtype = torch.bfloat16

    if args.impl == "reference":
        mod = load_reference()
    else:
        sys.path.insert(0, ROOT)
        import ring_flash_attn_b200 as mod
    fn = getattr(mod, f"zigzag_ring_flash_attn_{api}_func")

    torch.manual_seed(1234 + rank)
    if api == "qkvpacked":
        host_in = [torch.randn(1, tokens, 3, hq, d, dtype=dtype).pin_memory()]
    else:
        host_in = [torch.randn(1, tokens, hq, d, dtype=dtype).pin_memory(),
                   torch.randn(1, tokens, 2, hkv, d, dtype=dtype).pin_memory()]
    dev_in = [t.to(dev).requires_grad_(True) for t in host_in]
    dout = torch.randn(1, tokens, hq, d, dtype=dtype, device=dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    loss_host = torch.zeros(1, dtype=torch.float32).pin_memory()
    h2d_bytes = sum(t.numel() * t.element_size() for t in host_in)

    def step(inputs):
        if args.mode == "fwd":
            with torch.no_grad():
                return fn(*inputs, causal=True)
        for t in inputs:
            t.grad = None
        out = fn(*inputs, causal=True)
        out.backward(dout)
        return out

    def e2e_step():
        ins = [h.to(dev, non_blocking=True).requires_grad_(args.mode != "fwd") for h in host_in]
        out = step(ins)
        loss_host.copy_(out.float().mean().reshape(1), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return float(loss_host[0])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(run, steps, warmup):
        for _ in range(warmup):
            run()
        barrier()
        evs = []
        for _ in range(steps):
            last.clear()  # the previous step's result is released before this step allocates its own
            flush.fill_(1)  # evict L2 between timed iterations (outside the events)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            last.append(run())
            b.record()
            evs.append((a, b))
        barrier()
        per = sorted(a.elapsed_time(b) for a, b in evs)
        t = torch.tensor([sum(per) / steps, statistics.median(per), per[0], per[-1]], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        stats.update(mean=float(t[0]), median=float(t[1]), min=float(t[2]), max=float(t[3]))
        # the MEDIAN step (max over ranks) is the reported time: one NCCL / clock outlier in K steps must not
        # move the headline in either direction; mean / min / max stay in ms_per_step_stats
        return float(t[1])

    stats = {}
    last = []  # what the last timed step returned
    launches = None
    if args.impl == "ours":
        from ring_flash_attn_b200.ops import cuda_ext

        counter = cuda_ext.launch_counter()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    warm = args.warmup  # exactly what the caller asked for (the driver passes W >= 3)
    check = None
    if args.check and args.impl == "ours" and args.mode == "fwd_bwd":
        check = run_check(torch, fn, api, dev_in, dout, dist.group.WORLD if world > 1 else None)
    for _ in range(warm):
        step(dev_in)
    if args.impl == "ours":
        counter.reset()
    ms = timed(lambda: step(dev_in), args.steps, 0)
    step_stats = dict(stats)
    if args.impl == "ours":
        launches = counter.value
    dumped = None
    if args.dump_outputs:
        arrays = {"out": last[0]}
        if args.mode == "fwd_bwd":
            arrays.update(zip(["dqkv"] if api == "qkvpacked" else ["dq", "dkv"], (t.grad for t in dev_in)))
        dumped = sample_rows(torch, arrays, world)
        del arrays
    last.clear()
    e2e = None
    if not args.no_e2e:
        pipeline = "serial copy -> compute"
        run_e2e = e2e_step
        if os.environ.get("RFA_BENCH_E2E_PREFETCH", "1") == "1":
            try:
                run_e2e = PrefetchedE2E(torch.cuda, torch, dev, host_in, step, loss_host, args.mode != "fwd")
                run_e2e()  # one untimed step proves the pipeline works on this box before it is timed
                pipeline = "double-buffered prefetch on a side stream (copy of step i+1 under compute of step i)"
            except Exception as exc:  # noqa: BLE001 - never lose the benchmark line over the input pipeline
                run_e2e = e2e_step
                pipeline = f"serial copy -> compute (prefetch unavailable: {type(exc).__name__})"
        try:
            e2e_ms = timed(run_e2e, args.steps, warm)
        except Exception as exc:  # noqa: BLE001 - fall back to the serial loop rather than lose the line
            if run_e2e is e2e_step:
                raise
            pipeline = f"serial copy -> compute (prefetch failed while timing: {type(exc).__name__})"
            e2e_ms = timed(e2e_step, args.steps, warm)
        e2e = {"value": 1000.0 / e2e_ms, "unit": "iter/s", "ms_per_step": e2e_ms,
               "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4, "input_pipeline": pipeline}
    clocks = sampler.stop() if rank == 0 else None
    if dumped is not None:
        import numpy as np

        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ("" if world == 1 else f"_rank{rank}") + ".npy"), a)

    if rank == 0:
        value = 1000.0 / ms
        # causal attention FLOPs of the whole job: fwd 4*S^2*H*D/2, bwd 2.5x
        S = tokens * world
        fwd_flops = 2.0 * S * S * hq * d
        flops = fwd_flops * (3.5 if args.mode == "fwd_bwd" else 1.0)
        pub = PUBLISHED.get((args.config, world)) if args.mode == "fwd_bwd" else None
        line = {
            "metric": f"zigzag_ring_flash_attn_{api}_func {args.mode} iter/s",
            "value": value, "unit": "iter/s", "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": ms, "ms_per_step_stats": step_stats, "higher_is_better": True, "scaling": scaling,
            "vs_baseline": (value / pub) if pub else None, "dtype": "bf16", "data": "synthetic",
            "impl": args.impl,
            "config": {"model": "attention op (Llama-style heads)", "global_batch": 1, "seq_len": S,
                       "tokens_per_gpu": tokens, "nheads_q": hq, "nheads_kv": hkv, "head_dim": d, "causal": True,
                       "parallelism": f"cp{world}-zigzag", "api": f"zigzag_ring_flash_attn_{api}_func",
                       "name": args.config, "l2": "flushed with a 256 MiB write between timed steps"},
            "tflops_per_gpu": flops / world / (ms * 1e-3) / 1e12,
            "clocks": clocks,
        }
        if e2e is not None:
            line["e2e"] = e2e
        if launches is not None:
            line["gpu_launches"] = launches
        if check is not None:
            line["check"] = check
        print(json.dumps(line))
    if dist.is_initialized():
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
