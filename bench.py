#!/usr/bin/env python
"""Headline benchmark: sequence-parallel causal attention throughput (aggregate TFLOPS over N GPUs).

Contract (see task brief): ``python bench.py --gpus N --steps K --warmup W [--impl reference]`` prints
ONE JSON line on rank 0.  For N > 1 it is launched under torchrun (RANK/LOCAL_RANK/WORLD_SIZE env).

Config = BASELINE.json config 3 ("pure ring path") generalised over N:
  LongContextAttention(ring_impl_type="zigzag"), ulysses=1, ring=N, global seq 256K, h=8, d=128, bf16,
  causal, B=1, strong scaling (global problem fixed, each rank owns S/N tokens).
Both arms (ours / the unmodified reference from baseline/_ref with flash-attn 2.8.3 + NCCL) run the
same module API, the same shapes, the same timing harness.

value        device-timed (CUDA events, max over ranks) attention TFLOPS with inputs resident on device
e2e.value    same metric through the public API including, every step, the H2D copy of that step's
             q/k/v shards from pinned host memory and a D2H read of a scalar result
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


PRESETS = {
    2: dict(seq=32 * 1024, heads=32, ulysses=8, ring_impl="basic"),
    3: dict(seq=256 * 1024, heads=8, ulysses=1, ring_impl="zigzag"),
    4: dict(seq=128 * 1024, heads=32, kv_heads=4, ulysses=2, ring_impl="zigzag", window=8192),
    5: dict(seq=64 * 1024, heads=16, ulysses=4, ring_impl="zigzag", qkvpacked=True),
}


DUMP_BYTES = 64 * 10**6      # --dump-outputs: at most this many bytes of .npy files in all


def _positive(s):
    n = int(s)
    if n < 1:
        raise argparse.ArgumentTypeError(f"must be >= 1, got {n}")
    return n


def parse(argv=None):
    argv = list(sys.argv[1:] if argv is None else argv)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=_positive, default=5, help="timed steps (each timed loop runs exactly this many)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default=os.environ.get("LCA_BENCH_MODE", "fwdbwd"), choices=["fwd", "fwdbwd"])
    ap.add_argument("--seq", type=int, default=256 * 1024, help="GLOBAL sequence length")
    ap.add_argument("--heads", type=int, default=8)
    ap.add_argument("--kv-heads", type=int, default=0)
    ap.add_argument("--head-dim", type=int, default=128)
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--ulysses", type=int, default=1)
    ap.add_argument("--ring-impl", default="zigzag", choices=["basic", "zigzag", "strip"])
    ap.add_argument("--no-causal", action="store_true")
    ap.add_argument("--backend", default=None, help="ours: auto|fused|collective")
    ap.add_argument("--window", type=int, default=-1, help="sliding window (left) in tokens; -1 = none (BASELINE config 4)")
    ap.add_argument("--no-comm-probe", action="store_true",
                    help="skip the compute-only re-run that yields exposed_comm_ms (ours, N > 1; outside the timed regions)")
    ap.add_argument("--device", default="cuda", choices=["cuda", "cpu"],
                    help="cpu = control-flow dry run for the CPU test-suite (gloo, PyTorch engine, host timers); "
                         "numbers from it are meaningless")
    ap.add_argument("--qkvpacked", action="store_true", help="LongContextAttentionQKVPacked (BASELINE config 5; MHA only)")
    ap.add_argument("--config", type=int, default=0, choices=[0, 2, 3, 4, 5],
                    help="BASELINE.json config preset (2: pure Ulysses S=32K h=32; 3: pure ring zigzag S=256K h=8 [the default]; "
                         "4: U=2 x ring zigzag GQA kv=4 S=128K window; 5: U=4 x ring qkvpacked S=64K h=16); explicit flags win")
    ap.add_argument("--fp8", action="store_true", help="ours: e4m3 block-scaled forward (config 5); backward stays bf16")
    ap.add_argument("--no-check", action="store_true", help="skip the fp32 sampled-row correctness check after the timed regions")
    ap.add_argument("--configs", default="", help="comma-separated BASELINE config ids: run them all in ONE process group "
                    "(one JSON line per config x mode; saves the spawn + NCCL bootstrap of separate launches)")
    ap.add_argument("--modes", default="", help="with --configs: comma-separated modes (fwd,fwdbwd); default --mode")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last timed step returned to its caller (out; dq, dk, dv "
                         "in fwdbwd mode) as DIR/<name>.npy in float32, stacked over ranks; a seeded sample of token "
                         "rows when the whole would exceed 64 MB.  The inputs depend only on the arguments, so two "
                         "builds can be compared output for output")
    a = ap.parse_args(argv)
    if a.dump_outputs and a.configs:
        ap.error("--dump-outputs writes one configuration; it cannot be combined with --configs")
    if a.config:
        given = {x.split("=")[0].lstrip("-").replace("-", "_") for x in argv if x.startswith("--")}
        for key, val in PRESETS[a.config].items():
            if key not in given:
                setattr(a, key, val)
    return a


class ClockSampler:
    """Samples nvidia-smi SM clocks / throttle reasons of this rank's GPU during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.samples, self._stop, self._t = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 6:
                    self.samples.append(parts)
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(0.15)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        clocks = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        mx = max((int(s[1]) for s in self.samples if s[1].isdigit()), default=0)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": clocks[len(clocks) // 2] if clocks else None, "sm_max_mhz": mx or None,
                "reasons": reasons, "samples": len(clocks)}


class _HostCuda:
    """Stand-in for the ``torch.cuda`` calls of this script in ``--device cpu`` dry runs (tests/test_bench_cpu.py)."""

    class Event:
        def __init__(self, enable_timing=False):
            self.t = 0.0

        def record(self, stream=None):
            import time
            self.t = time.perf_counter()

        def elapsed_time(self, other):
            return max((other.t - self.t) * 1e3, 1e-6)

    class Stream:
        def __init__(self, device=None):
            pass

        def wait_event(self, ev):
            pass

    @staticmethod
    def stream(s):
        import contextlib
        return contextlib.nullcontext()

    @staticmethod
    def current_stream(device=None):
        return _HostCuda.Stream()

    @staticmethod
    def synchronize(device=None):
        pass

    @staticmethod
    def set_device(i):
        pass


def dump_outputs(path, arrays, dist, rank, budget=DUMP_BYTES):
    """Writes every (B, S/N, H, D) shard of ``arrays`` (name -> tensor) as ``path/<name>.npy``: float32, shape
    (N, B, rows, H, D), rank r's shard at index r.  ``dist`` is None in a single process.  When all shards of all
    arrays exceed ``budget`` bytes, the same seeded sample of local token rows (sorted) is taken from each of them.
    Every rank must call this; rank 0 writes.  Returns a description of what was written."""
    import numpy as np
    import torch

    world = dist.get_world_size() if dist is not None else 1
    Sl = next(iter(arrays.values())).shape[1]
    row_bytes = 4 * world * sum(t[:, 0].numel() for t in arrays.values())
    n = min(Sl, (budget - 1024 * len(arrays)) // row_bytes)          # 1 KiB per file covers the .npy header
    rows = torch.arange(Sl) if n == Sl else torch.randperm(Sl, generator=torch.Generator().manual_seed(0))[:n].sort().values
    if rank == 0:
        os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        s = t.detach()[:, rows.to(t.device)].float().contiguous()
        parts = [s]
        if dist is not None:
            parts = [torch.empty_like(s) for _ in range(world)]
            dist.all_gather(parts, s)
        if rank == 0:
            np.save(os.path.join(path, name + ".npy"), torch.stack(parts).cpu().numpy())
    return {"dir": path, "arrays": list(arrays), "dtype": "float32", "layout": "(rank, batch, row, head, dim)",
            "rows_per_rank": int(n), "local_seq": int(Sl), "row_sample_seed": None if n == Sl else 0}


def main():
    a0 = parse()
    import torch
    import torch.distributed as dist
    on_cpu = a0.device == "cpu"
    cu = _HostCuda if on_cpu else torch.cuda          # every CUDA runtime call below goes through `cu`

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a0.gpus:
        if world == 1 and a0.gpus > 1:
            raise SystemExit("launch with torchrun for --gpus > 1")
    cu.set_device(local_rank)
    dev = torch.device("cpu") if on_cpu else torch.device("cuda", local_rank)

    if a0.impl == "reference":
        ref_dir = os.path.join(ROOT, "baseline", "_ref")
        if not os.path.isdir(os.path.join(ref_dir, "yunchang")):
            print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref/yunchang missing (pip install --target failed)"}))
            return
        sys.path.insert(0, ref_dir)
    need_dist = world > 1 or a0.impl == "reference"
    if need_dist:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29533")
        if on_cpu:
            dist.init_process_group("gloo", rank=rank, world_size=world)
        else:
            dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    ctx = dict(torch=torch, dist=dist, on_cpu=on_cpu, cu=cu, world=world, rank=rank, local_rank=local_rank, dev=dev,
               need_dist=need_dist)
    runs = [a0]
    if a0.configs:
        base = [x for x in sys.argv[1:]]
        modes = [m for m in (a0.modes.split(",") if a0.modes else [a0.mode]) if m]
        runs = [parse(base + ["--config", c, "--mode", m]) for c in a0.configs.split(",") if c for m in modes]
    bad = False
    for a in runs:
        ok = run_config(a, ctx)
        bad = bad or ok is False
    if need_dist:
        dist.destroy_process_group()
    if bad:
        raise SystemExit(3)          # a wrong answer must not look like a benchmark result


def run_config(a, ctx):
    """One benchmark configuration inside an initialised process group; prints ONE JSON line on rank 0.
    Returns False when the correctness check of our arm failed."""
    torch, dist, on_cpu, cu = ctx["torch"], ctx["dist"], ctx["on_cpu"], ctx["cu"]
    world, rank, local_rank, dev, need_dist = ctx["world"], ctx["rank"], ctx["local_rank"], ctx["dev"], ctx["need_dist"]
    N = world
    U = min(a.ulysses, N)
    R = N // U
    B, S, H, D = a.batch, a.seq, a.heads, a.head_dim
    Hkv = a.kv_heads or H
    causal = not a.no_causal
    Sl = S // N
    assert S % (2 * N) == 0
    dtype = torch.bfloat16

    if a.impl == "reference":
        try:
            import yunchang
            from yunchang import LongContextAttention, set_seq_parallel_pg
            from yunchang.kernels import AttnType
        except Exception as e:  # noqa: BLE001
            if rank == 0:
                print(json.dumps({"impl": "reference", "unavailable": f"import yunchang failed: {type(e).__name__}: {str(e)[:120]}"}))
            return
        set_seq_parallel_pg(U, R, rank, world)
        if a.qkvpacked:
            from yunchang import LongContextAttentionQKVPacked
            attn = LongContextAttentionQKVPacked(ring_impl_type=a.ring_impl, attn_type=AttnType.FA)
        else:
            attn = LongContextAttention(ring_impl_type=a.ring_impl, attn_type=AttnType.FA)
        launches = lambda: 0
        native_ok = None
    else:
        import lca_b200
        from lca_b200 import LongContextAttention, set_seq_parallel_pg
        from lca_b200.ops import native

        set_seq_parallel_pg(U, R, rank, world)
        extra = {}
        if on_cpu:                       # dry run: PyTorch engine over gloo
            from lca_b200.kernels import AttnType
            extra = dict(attn_type=AttnType.TORCH)
        if a.qkvpacked:
            from lca_b200 import LongContextAttentionQKVPacked
            attn = LongContextAttentionQKVPacked(ring_impl_type=a.ring_impl, backend=a.backend, **extra)
        else:
            attn = LongContextAttention(ring_impl_type=a.ring_impl, backend=a.backend, **extra)
        launches = lambda: native.LAUNCHES
        native_ok = native.available()
        assert native_ok or on_cpu, "native sm_100a extension not available on this GPU box"

    # synthetic shards, generated on host in pinned memory (this rank's S/N tokens)
    g = torch.Generator().manual_seed(1234 + rank)
    host = [torch.randn(B, Sl, h, D, generator=g, dtype=torch.float32).to(dtype) for h in (H, Hkv, Hkv)]
    if not on_cpu:
        host = [t.pin_memory() for t in host]
    host_do = torch.randn(B, Sl, H, D, generator=g, dtype=torch.float32).to(dtype)
    if not on_cpu:
        host_do = host_do.pin_memory()
    need_grad = a.mode == "fwdbwd"

    def to_dev(non_blocking=True):
        """This step's inputs: q, k, v (and the upstream gradient dO in fwd+bwd mode) from pinned host memory."""
        ts = [t.to(dev, non_blocking=non_blocking, copy=True) for t in host]     # copy: fresh leaves on cpu too
        if need_grad:
            ts = [t.requires_grad_() for t in ts]
            ts.append(host_do.to(dev, non_blocking=non_blocking))
        return ts

    dout = host_do.to(dev)
    flush = torch.empty((1 if on_cpu else 256) * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2

    kw = dict(causal=causal)
    if a.window >= 0:
        kw["window_size"] = (a.window, 0 if causal else a.window)

    def call(q, k, v):
        if a.qkvpacked:
            return attn(torch.stack([q, k, v], dim=2), **kw)      # (B, S/P, 3, H, D)
        return attn(q, k, v, **kw)

    def step(q, k, v, do=None):
        if need_grad:
            out = call(q, k, v)
            out.backward(dout if do is None else do)
            return out
        with torch.no_grad():
            return call(q, k, v)

    def barrier():
        if need_dist and world > 1:
            dist.barrier()
        cu.synchronize()

    # ------------------------------------------------------------------ device-resident timing
    q, k, v = to_dev(False)[:3]
    for _ in range(max(a.warmup, 3)):
        step(q, k, v)
        flush.fill_(1)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = launches()
    e0, e1 = cu.Event(enable_timing=True), cu.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        step(q, k, v)
        flush.fill_(1)       # evict inputs/outputs from L2 between timed iterations
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1) / a.steps
    n_launch = (launches() - l0) // max(a.steps, 1)

    # ------------------------------------------------------------------ end-to-end timing
    copy_stream = cu.Stream(device=dev)
    cur = cu.current_stream(dev)

    def prefetch():
        with cu.stream(copy_stream):
            ts = to_dev(True)
            ev = cu.Event()
            ev.record(copy_stream)
        return ts, ev

    results = []

    def run_pipelined(n):
        """Returns the last step's inputs and output."""
        nxt = prefetch()
        for i in range(n):
            ts, ev = nxt
            cur.wait_event(ev)
            for t in ts:
                if not on_cpu:
                    t.record_stream(cur)
            if i + 1 < n:
                nxt = prefetch()          # H2D of step i+1 overlaps the attention of step i
            out = step(*ts)
            results.append(float(out.float().mean().item()))     # D2H read of the step's result
        return ts, out

    run_pipelined(3)        # warm the pipelined path with the same allocation pattern (two input sets in flight)
    cu.synchronize(dev)
    barrier()
    t_ev0, t_ev1 = cu.Event(enable_timing=True), cu.Event(enable_timing=True)
    t_ev0.record()
    last_in, last_out = run_pipelined(a.steps)
    t_ev1.record()
    barrier()
    clocks = sampler.stop()
    ms_e2e = t_ev0.elapsed_time(t_ev1) / a.steps

    if need_dist and world > 1:
        t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = float(t[0]), float(t[1])

    # The last timed step takes fresh leaf tensors from the same host inputs as every other step, so its gradients
    # are that step's alone (the device-resident loop accumulates into q/k/v.grad across steps).
    dumped = None
    if a.dump_outputs:
        arrays = {"out": last_out}
        if need_grad:
            arrays.update(dq=last_in[0].grad, dk=last_in[1].grad, dv=last_in[2].grad)
        dumped = dump_outputs(a.dump_outputs, arrays, dist if world > 1 else None, rank)
    del last_in, last_out

    # ------------------------------------------------------------------ exposed communication (ours, N > 1)
    # The same tcgen05 kernels on the same per-rank problem (this rank's ring block of queries against all S keys,
    # its head slice) with every operand already local: no pushes, no arrival flags, no NVLink traffic.  The
    # difference to the fused step time is the communication the fused kernels failed to hide.
    comm_probe = None
    if a.impl == "ours" and world > 1 and not a.no_comm_probe:
        local_ms = float("nan")
        try:
            from lca_b200.ops.attention import AttnParams, attn_block_bwd, attn_block_fwd
            from lca_b200.parallel.layout import Seg, ring_positions
            Sr, Hl, Hkvl = U * Sl, H // U, max(Hkv // U, 1)
            gq = torch.Generator(device=dev)
            gq.manual_seed(99 + rank)
            qb = torch.randn(B, Sr, Hl, D, generator=gq, device=dev, dtype=torch.float32).to(dtype)
            dob = torch.randn(B, Sr, Hl, D, generator=gq, device=dev, dtype=torch.float32).to(dtype)
            kf = torch.randn(B, S, Hkvl, D, generator=gq, device=dev, dtype=torch.float32).to(dtype)
            vf = torch.randn(B, S, Hkvl, D, generator=gq, device=dev, dtype=torch.float32).to(dtype)
            win = (a.window, 0 if causal else a.window) if a.window >= 0 else (-1, -1)
            pp = AttnParams.make(qb, None, causal, win)
            q_pos = ring_positions(a.ring_impl, rank // U, R, Sr)
            k_pos = (Seg(0, S, 1),)

            def local_step():
                o, l = attn_block_fwd(qb, kf, vf, q_pos, k_pos, pp)        # native tcgen05 kernels on a GPU box
                if need_grad:
                    attn_block_bwd(dob, qb, kf, vf, o, l, q_pos, k_pos, pp)

            for _ in range(2):
                local_step()
            cu.synchronize(dev)
            n_probe = max(1, min(a.steps, 5))
            c0, c1 = cu.Event(enable_timing=True), cu.Event(enable_timing=True)
            c0.record()
            for _ in range(n_probe):
                local_step()
                flush.fill_(1)
            c1.record()
            cu.synchronize(dev)
            local_ms = c0.elapsed_time(c1) / n_probe
            del qb, dob, kf, vf
        except Exception as e:  # noqa: BLE001 - the probe must never cost the headline number
            comm_probe = {"error": f"{type(e).__name__}: {str(e)[:160]}"}
        t = torch.tensor([local_ms if local_ms == local_ms else -1.0], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if comm_probe is None and float(t[0]) > 0:
            comm_probe = {"compute_only_ms": round(float(t[0]), 4), "exposed_comm_ms": round(ms - float(t[0]), 4),
                          "how": "same kernels, same per-rank problem, all operands local (no NVLink); max over ranks"}

    # ------------------------------------------------------------------ correctness (outside every timer)
    # One more step on the device-resident shards; the last kv head (and its query heads) of out / dq / dk / dv is
    # gathered into natural token order and compared on sampled rows / columns with the chunked fp32 oracle
    # (lca_b200/ops/sampled_oracle.py) evaluated on the gathered K/V.  Every rank checks its own sample.
    check = None
    if not a.no_check and not on_cpu:
        try:
            from lca_b200.ops.sampled_oracle import head_oracle, rel_err
            from lca_b200.parallel.layout import canonical_variant, gather_global
            variant = canonical_variant(a.ring_impl)
            qc, kc, vc = (t.detach().clone().requires_grad_(need_grad) for t in (q, k, v))
            oc = call(qc, kc, vc) if need_grad else step(qc, kc, vc)
            if need_grad:
                oc.backward(dout)
            G, hk = H // Hkv, Hkv - 1

            def glob(t):
                t = t.detach().contiguous()
                if world == 1:
                    return t
                parts = [torch.empty_like(t) for _ in range(world)]
                dist.all_gather(parts, t)
                return gather_global(variant, parts, R, U)

            hs = slice(hk * G, (hk + 1) * G)
            gq, gk, gv, go = glob(q[:, :, hs]), glob(k[:, :, hk:hk + 1]), glob(v[:, :, hk:hk + 1]), glob(oc[:, :, hs])
            gdo = glob(dout[:, :, hs]) if need_grad else None
            gs = torch.Generator().manual_seed(4321 + rank)
            n_rows, n_cols = 128, (64 if need_grad else 0)
            rows = torch.randint(0, S, (n_rows,), generator=gs)
            rows[0], rows[1] = 0, S - 1
            cols = None
            if n_cols:
                cols = torch.randint(0, S, (n_cols,), generator=gs)
                cols[0], cols[1] = 0, S - 1
            win = (a.window, 0 if causal else a.window) if a.window >= 0 else (-1, -1)
            ref = head_oracle(gq[0], gk[0, :, 0], gv[0, :, 0], gdo[0] if need_grad else None, rows, cols, causal=causal,
                              window=win, chunk=2048)
            rows_d = rows.to(dev)
            errs = {"max_err_out": float((go[0, rows_d].float() - ref["out"]).abs().max())}
            if need_grad:
                cols_d = cols.to(dev)
                errs["max_rel_err_dq"] = rel_err(glob(qc.grad[:, :, hs])[0, rows_d], ref["dq"])
                errs["max_rel_err_dk"] = rel_err(glob(kc.grad[:, :, hk:hk + 1])[0, cols_d, 0], ref["dk"])
                errs["max_rel_err_dv"] = rel_err(glob(vc.grad[:, :, hk:hk + 1])[0, cols_d, 0], ref["dv"])
            t = torch.tensor([errs.get("max_err_out", 0.0), errs.get("max_rel_err_dq", 0.0), errs.get("max_rel_err_dk", 0.0),
                              errs.get("max_rel_err_dv", 0.0)], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            vals = [float(x) for x in t]
            ok = vals[0] < 2e-2 and all(x < 3e-2 for x in vals[1:]) and all(x == x for x in vals)
            check = {"max_err_out": round(vals[0], 5), "ok": bool(ok), "rows_per_rank": n_rows, "cols_per_rank": n_cols,
                     "head": int(hk), "oracle": "fp32 chunked softmax on gathered K/V (ops/sampled_oracle.py)"}
            if need_grad:
                check.update({"max_rel_err_dq": round(vals[1], 5), "max_rel_err_dk": round(vals[2], 5),
                              "max_rel_err_dv": round(vals[3], 5)})
            if a.window >= 0 and a.impl == "reference":
                check["note"] = "the reference applies the window per ring block without global offsets (BASELINE.md section 7)"
            del gq, gk, gv, go, gdo, ref
        except Exception as e:  # noqa: BLE001
            check = {"ok": False, "error": f"{type(e).__name__}: {str(e)[:200]}"}

    staging = None
    if a.impl == "ours" and world > 1:
        try:
            from lca_b200.parallel import fused_engine as _fe
            engs = [e for e in _fe._ENGINES.values() if e is not None]
            if engs:
                staging = {"slab_bytes_per_rank": int(engs[0].slab_bytes), "push_ctas": int(engs[0].n_comm)}
        except Exception:  # noqa: BLE001
            pass

    flops = 4.0 * B * H * S * S * D * (0.5 if causal else 1.0)
    if need_grad:
        flops *= 3.5
    tflops = flops / (ms * 1e-3) / 1e12
    tflops_e2e = flops / (ms_e2e * 1e-3) / 1e12
    h2d = sum(t.numel() * t.element_size() for t in host) + (host_do.numel() * host_do.element_size() if need_grad else 0)
    if rank == 0:
        print(json.dumps({
            "metric": "attention_tflops_" + ("fwd_bwd" if need_grad else "fwd"),
            "value": round(tflops, 2), "unit": "TFLOPS", "n_gpus": N, "steps": a.steps, "warmup": max(a.warmup, 3),
            "ms_per_step": round(ms, 4), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic (randn q/k/v shards, no weights in this op)",
            "impl": a.impl,
            "config": {"model": "LongContextAttention(ring_impl_type=%s)" % a.ring_impl, "global_batch": B,
                       "seq_len": S, "heads": H, "kv_heads": Hkv, "head_dim": D, "causal": causal,
                       "parallelism": f"ulysses{U}xring{R}", "mode": a.mode, "window": a.window, "qkvpacked": a.qkvpacked,
                       "l2": "256 MiB flush write between timed iterations; per-rank q+k+v+o also exceed L2",
                       "native_kernels": native_ok},
            "clocks": clocks,
            "e2e": {"value": round(tflops_e2e, 2), "unit": "TFLOPS", "ms_per_step": round(ms_e2e, 4),
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4},
            "gpu_launches": int(n_launch * a.steps) if a.impl == "ours" else None,
            "comm": comm_probe,
            "config_id": a.config or 3,
            "check": check,
            "staging": staging,
            "outputs": dumped,
        }))
    del attn
    if a.impl == "ours" and check is not None and not check.get("ok", False):
        return False
    return True


if __name__ == "__main__":
    main()
