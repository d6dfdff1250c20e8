#!/usr/bin/env python
"""bench.py -- throughput of the NAM inference hot path on B200 (one JSON line, driver contract).

Workload (BASELINE.json metric): wavenet_a1_standard.nam, batch 4096 independent 48 kHz streams per GPU,
float32.  A "step" is ONE pass of the hot path over one batch of synthetic input: 4096 streams x
`--frames` frames (default 4096), state carried across steps in HBM exactly like successive
DSP::process() calls.  Weak scaling: every GPU runs its own 4096 streams (no data-path collective; the
streams are independent, SURVEY.md 8e).

  value      Msamples/s, whole job, inputs/outputs resident in HBM, CUDA-event timed, max over ranks
  e2e        same metric through the public host API (nam_b200_process_f32 with pinned host buffers:
             H2D + kernel + D2H inside the timed region)
  roofline   the fused kernel against the FP32 FMA pipe (self-measured FFMA2 peak) -- the binding roof
             for this path (DESIGN.md "Roofline") -- plus HBM / tensor fractions for context
  cpu_baseline  the CPU restatement (oracle/, "port") on all host cores, bounded sample
  --impl reference   times that CPU port as the reference arm (the reference itself cannot be built
             here: Eigen is an un-vendored submodule, see DESIGN.md)

Nothing here reads /root/reference.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "Msamples/sec (48kHz RTF) wavenet_a1_standard.nam, batch 4096, 1/2/4/8 GPU vs Eigen CPU"
MODEL = "wavenet_a1_standard"
CPU_BLOCK = 64  # AUDIO_BUFFER_SIZE of tools/benchmodel.cpp:18


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=4096, help="streams per GPU")
    ap.add_argument("--frames", type=int, default=4096, help="frames per stream per step")
    ap.add_argument("--model", default=MODEL)
    ap.add_argument("--tanh", default="fast", choices=["fast", "exact"],
                    help="fast = tools/benchmodel.cpp default (enable_fast_tanh); exact = library default")
    ap.add_argument("--ctas-per-sm", type=int, default=0)
    ap.add_argument("--geometry", type=int, default=0, help="0 default, 1 = FP32 kernel 128-thread CTAs, 2 = FP32 kernel 256-thread CTAs, 3 = tensor-core kernel")
    ap.add_argument("--jit", type=int, default=0, help="model-specialised kernel: 0 = library default (on at batch >= 256), 1 = required, 2 = off")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the quick batch-1/256, A2, LSTM, a2_max lines")
    ap.add_argument("--no-gather", action="store_true",
                    help="N > 1: skip the second timed pass that all-gathers every step's outputs over NCCL")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/y.npy (DIR/y_rank<r>.npy at N > 1), float32, "
                         "streams x frames; above 64 MB in all, a fixed seeded choice of streams in ascending order")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    if args.dump_outputs and args.steps < 1:
        ap.error("--dump-outputs writes the outputs of the last timed step: --steps must be at least 1")
    return args


# ---------------------------------------------------------------------------------------------------
def load_peaks() -> dict:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            d = json.loads(p.read_text())
            d["_source"] = "measured"
            return d
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "_source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows: list[list[str]] = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                for line in out.strip().splitlines():
                    self.rows.append([c.strip() for c in line.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)

    def summary(self) -> dict:
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except Exception:
                continue
            for name, val in zip(names, r[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def fixtures():
    from tests import nam_fixtures as fx

    return fx


def cpu_port_lib():
    """The CPU restatement built -march=native on THIS box (falls back to the in-tree x86-64-v3 build)."""
    from oracle import oracle

    oracle.build()
    native = oracle.build_native_fast(tempfile.mkdtemp(prefix="nam_oracle_"))
    if native is not None:
        try:
            return oracle.load_lib(path=native), "-O3 -march=native -ffast-math"
        except OSError:
            pass
    return oracle.load_lib("fast"), "-O3 -march=x86-64-v3 -ffast-math"


def host_threads() -> int:
    """Threads this process may really use: cpu_count, the affinity mask and the cgroup CPU quota."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except AttributeError:
        pass
    try:
        quota, period = Path("/sys/fs/cgroup/cpu.max").read_text().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return max(n, 1)


def best_cpu_port(nam: dict, fast_tanh: bool, frames: int, streams_per_thread: int) -> tuple[float, float, int, int]:
    """The CPU port at full, half and quarter thread counts (SMT siblings and shared caches often make fewer
    threads faster on the 196 KB-per-stream working set); returns the best (Msamples/s, seconds, threads, streams)."""
    t_all = host_threads()
    best = (0.0, 0.0, t_all, 0)
    for threads in sorted({t_all, max(t_all // 2, 1), max(t_all // 4, 1)}, reverse=True):
        streams = streams_per_thread * threads
        v, secs = time_cpu_port(nam, fast_tanh, frames, streams, threads)
        if v > best[0]:
            best = (v, secs, threads, streams)
    return best


def time_cpu_port(nam: dict, fast_tanh: bool, frames: int, streams: int, threads: int, reps: int = 1) -> tuple[float, float]:
    """Returns (Msamples/s, seconds per rep) of the CPU port on `threads` host threads."""
    from oracle import oracle

    lib, _ = cpu_port_lib()
    fx = fixtures()
    proto = oracle.OracleModel.from_dict(nam, fast_tanh=fast_tanh, lib=lib)
    proto.reset(48000.0, CPU_BLOCK)  # the reference tools' protocol: Reset(sr, 64), 64-frame process() calls
    pool = oracle.OracleBatch(proto, streams)  # one DSP instance per stream, created outside the timed region
    x = fx.synthetic_batch(streams, frames, seed=99)
    y = np.empty_like(x)
    pool.process(np.ascontiguousarray(x[:, :CPU_BLOCK * 4]), None, CPU_BLOCK, threads)  # warm-up
    best = float("inf")
    for _ in range(reps):
        t0 = time.perf_counter()
        pool.process(x, y, CPU_BLOCK, threads)
        best = min(best, time.perf_counter() - t0)
    pool.close()
    return streams * frames / best / 1e6, best


def time_reference_build(nam: dict, fast_tanh: bool, frames: int, streams: int, threads: int, reps: int = 1):
    """(Msamples/s, seconds, variant) of the reference's OWN sources (oracle/_ref, -Ofast like tools/CMakeLists.txt:106,
    Eigen stand-in with in-place register-blocked products) under the benchmodel protocol, or None if not built."""
    from oracle import ref

    variant = ref.best_timed_variant()
    if variant is None:
        return None
    fx = fixtures()
    pool = ref.ReferencePool(nam, streams, fast_tanh, variant, CPU_BLOCK)
    x = fx.synthetic_batch(streams, frames, seed=99)
    y = np.empty_like(x)
    pool.process(np.ascontiguousarray(x[:, :CPU_BLOCK * 4]), np.empty((streams, CPU_BLOCK * 4), np.float32), threads)  # warm-up
    best = float("inf")
    for _ in range(reps):
        t0 = time.perf_counter()
        pool.process(x, y, threads)
        best = min(best, time.perf_counter() - t0)
    pool.close()
    return streams * frames / best / 1e6, best, variant


def cpu_arms(nam: dict, fast_tanh: bool, frames: int, streams_per_thread: int) -> dict:
    """Both CPU implementations of the path on this box's host cores, at the port's best thread count: the C restatement
    ("port") and the reference's own sources ("reference").  The FASTER one is the baseline the GPU is compared with."""
    v, secs, cores, streams = best_cpu_port(nam, fast_tanh, frames, streams_per_thread)
    _, flags = cpu_port_lib()
    out = {"port": {"value": v, "seconds": secs, "cores": cores, "streams": streams, "flags": f"gcc {flags}"}}
    try:
        r = time_reference_build(nam, fast_tanh, frames, streams, cores)
        if r is not None:
            out["reference"] = {"value": r[0], "seconds": r[1], "cores": cores, "streams": streams,
                                "flags": f"g++ -Ofast -march={'x86-64-v4' if r[2] == 'fast512' else 'x86-64-v3'} "
                                         "(tools/CMakeLists.txt:106), the unmodified reference NAM sources, Eigen stand-in"}
    except Exception as exc:  # the reference build is optional on the box
        out["reference_error"] = str(exc)[:200]
    kind = "reference" if out.get("reference", {}).get("value", 0.0) > v else "port"
    out["kind"] = kind
    return out


# ---------------------------------------------------------------------------------------------------
def run_reference(args) -> None:
    """--impl reference: the reference's CPU algorithm for the path on the host cores, same config/metric/unit.

    Two CPU implementations exist here: the C restatement (oracle/nam_oracle.c, "port") and the reference's own
    sources compiled against a stand-in for their missing Eigen submodule (oracle/_ref, validated bit-close against
    the port in tests/test_reference_build.py).  The stand-in evaluates every Eigen expression into a temporary, so
    the reference build runs ~5x slower than the port; timing THAT as "the reference" would flatter the GPU.  The
    line's value is therefore the faster one (the port, built -O3 -march=native -ffast-math like the reference's
    -Ofast Release build); the reference build's own rate is reported beside it."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    fx = fixtures()
    nam = fx.load_model(args.model)
    from oracle import oracle

    lib, flags = cpu_port_lib()
    fast = args.tanh == "fast"
    # pick the thread count once (short probe), then time exactly K steps at it
    _, _, cores, streams = best_cpu_port(nam, fast, 2048, 2)
    proto = oracle.OracleModel.from_dict(nam, fast_tanh=fast, lib=lib)
    proto.reset(48000.0, CPU_BLOCK)
    pool = oracle.OracleBatch(proto, streams)
    x = fx.synthetic_batch(streams, args.frames, seed=99)
    y = np.empty_like(x)
    for _ in range(max(args.warmup, 1)):
        pool.process(x, y, CPU_BLOCK, cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        pool.process(x, y, CPU_BLOCK, cores)
    dt = time.perf_counter() - t0
    pool.close()
    value = streams * args.frames * args.steps / dt / 1e6
    port_value = value
    sample = (f"{streams} of {args.batch} streams x {args.frames} frames per step in {CPU_BLOCK}-frame process() calls "
              f"(tools/benchmodel.cpp protocol), one instance per stream, {cores} threads (best of full/half/quarter "
              f"of the {host_threads()} usable), gcc {flags}")
    # the reference's own sources under the same protocol, same streams / threads / steps
    ref_build = None
    kind = "port"
    try:
        from oracle import ref

        variant = ref.best_timed_variant()
        if variant is not None:
            rpool = ref.ReferencePool(nam, streams, fast, variant, CPU_BLOCK)
            for _ in range(max(args.warmup, 1)):
                rpool.process(x, y, cores)
            t1 = time.perf_counter()
            for _ in range(args.steps):
                rpool.process(x, y, cores)
            d1 = time.perf_counter() - t1
            rpool.close()
            rv = streams * args.frames * args.steps / d1 / 1e6
            ref_build = {"value": rv, "unit": "Msamples/s", "cores": cores, "ms_per_step": d1 / args.steps * 1e3,
                         "what": f"oracle/_ref/{ref.lib_path(variant).name}: the unmodified reference sources, g++ -Ofast "
                                 f"-march={'x86-64-v4' if variant == 'fast512' else 'x86-64-v3'} (tools/CMakeLists.txt:106), "
                                 "Eigen stand-in with in-place register-blocked products (oracle/eigen_shim)"}
            if rv > value:  # the line carries the FASTER CPU implementation
                port_value, value, dt, kind = value, rv, d1, "reference"
                sample = sample.replace(f"gcc {flags}", ref_build["what"])
                ref_build["port_value"] = port_value
    except Exception as exc:  # the checker is optional on the box
        ref_build = {"unavailable": str(exc)[:200]}
    line = {
        "impl": "reference",
        "metric": metric_name(args),
        "value": value,
        "unit": "Msamples/s",
        "n_gpus": args.gpus,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": workload_config(args),
        "rtf_48k_aggregate": value * 1e6 / 48000.0,
        "cpu_baseline": {"value": value, "unit": "Msamples/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "port": {"value": port_value if kind == "reference" else value, "unit": "Msamples/s", "flags": f"gcc {flags}"},
        "reference_build": ref_build,
        "note": "two CPU implementations are timed on the same streams / threads / steps: the C restatement (oracle/nam_oracle.c, "
                "\"port\") and the reference's own sources compiled here (oracle/_ref, \"reference\"); the line's value is the "
                "faster one (cpu_baseline.kind)",
    }
    print(json.dumps(line), flush=True)


def metric_name(args) -> str:
    """BASELINE.json's metric; other models (secondary workloads) are named in it instead of a1_standard."""
    return METRIC if args.model == MODEL else METRIC.replace("wavenet_a1_standard.nam", f"{args.model}.nam")


def workload_config(args) -> dict:
    return {
        "workload": f"{args.model}.nam, {args.batch} independent 48 kHz streams per GPU x {args.frames} frames per step, "
                    f"float32, {args.tanh}-tanh regime, stateful (history carried across steps in HBM)",
        "streams_per_gpu": args.batch,
        "frames_per_step": args.frames,
        "tanh": args.tanh,
        "l2_policy": "working set per step (in+out+touched state) exceeds L2; no flush needed",
    }


DUMP_BYTES = 64 * 10**6  # --dump-outputs: at most this much in all, over every rank


def dump_outputs(out_dir: str, y, rank: int, world: int) -> None:
    """y (streams x frames, float32 on the device) -> out_dir/y.npy.  Where all ranks' outputs would exceed DUMP_BYTES,
    each rank keeps the same seeded choice of streams, so two runs with the same arguments write the same streams."""
    import torch

    streams, frames = y.shape
    keep = min(streams, DUMP_BYTES // (world * frames * y.element_size()))
    if keep < 1:
        raise SystemExit(f"bench.py: --dump-outputs: one stream of {frames} frames exceeds {DUMP_BYTES} bytes")
    rows = np.arange(streams) if keep == streams else np.sort(np.random.default_rng(0).choice(streams, keep, replace=False))
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / ("y.npy" if world == 1 else f"y_rank{rank}.npy"), y[torch.from_numpy(rows).to(y.device)].cpu().numpy())


def run_b200(args) -> None:
    import torch

    import neuralampmodelercore_b200 as nb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    fx = fixtures()
    nam = fx.load_model(args.model)
    B, n = args.batch, args.frames
    fast = args.tanh == "fast"

    model = nb.get_dsp(nam, batch=B, device=local_rank, fast_tanh=fast, ctas_per_sm=args.ctas_per_sm,
                       kernel_geometry=args.geometry, jit=args.jit)
    model.Reset(48000.0, n)
    jit_state, jit_note = model.jit_state, model.jit_note()
    flops_per_frame = model.flops_per_frame
    state_bytes = model.state_bytes_per_stream

    x_host = torch.from_numpy(fx.synthetic_batch(B, n, seed=1234 + rank)).pin_memory()
    y_host = torch.empty_like(x_host).pin_memory()
    x_dev = x_host.cuda(non_blocking=True)
    y_dev = torch.empty_like(x_dev)
    # a non-default stream: its handle is passed to the C ABI so kernels and the timing events share a stream
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)

    def step_device():
        model.process_batch_device(x_dev.data_ptr(), y_dev.data_ptr(), B, n, n, n, stream.cuda_stream)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput (value) ----
    for _ in range(args.warmup):
        step_device()
    barrier()
    launches0 = model.launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    with ClockSampler(local_rank) as clocks:
        ev[0].record(stream)
        for i in range(args.steps):
            step_device()
            ev[i + 1].record(stream)
        barrier()
    total_ms = ev[0].elapsed_time(ev[-1])
    step_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    launches = model.launch_count() - launches0
    t = torch.tensor([total_ms], device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    value = world * B * n * args.steps / (total_ms_max * 1e-3) / 1e6
    if args.dump_outputs:  # before the passes below write y_dev again
        dump_outputs(args.dump_outputs, y_dev, rank, world)

    # ---- end to end through the host API ----
    e2e = None
    if not args.no_e2e:
        xh, yh = x_host.numpy(), y_host.numpy()
        for _ in range(max(1, min(args.warmup, 3))):
            model.process_batch(xh, yh)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            model.process_batch(xh, yh)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        loss = float(np.abs(yh[0, :8]).sum())  # touch the result on the host
        e2e = {"value": world * B * n * args.steps / float(t.item()) / 1e6, "unit": "Msamples/s",
               "h2d_bytes_per_step": int(x_host.numel() * 4), "d2h_bytes_per_step": int(y_host.numel() * 4),
               "ms_per_step": float(t.item()) / args.steps * 1e3, "checksum": loss}

    # ---- N > 1: the same K steps again, now with the NCCL all-gather of every step's outputs (BASELINE.json config 5:
    # "batch sharded 4096/GPU, NCCL gather of output buffers").  The streams are independent, so the gather is the only
    # collective the path can have; it runs on a side stream and overlaps the NEXT step's kernel (outputs double-buffered),
    # the way a host that wants all outputs on every rank would drive it.  Timed like `value`: CUDA events, max over ranks.
    gather = None
    value_with_gather = None
    if dist is not None and not args.no_gather:
        # three output buffers: the persistent kernel holds every SM for the whole step, so the gather of step i only gets
        # SMs when step i+1's kernel drains; with two buffers step i+2 would then wait for that gather behind an idle GPU
        # (measured at N = 2: 11.01 ms per step against 10.39 + 0.19 for kernel + collective)
        NB = 3
        y2 = [y_dev] + [torch.empty_like(y_dev) for _ in range(NB - 1)]
        gathered = [torch.empty((world,) + tuple(y_dev.shape), dtype=y_dev.dtype, device="cuda") for _ in range(NB)]
        side = torch.cuda.Stream()
        done = [torch.cuda.Event() for _ in range(NB)]  # gather of buffer b finished (side stream)
        ready = torch.cuda.Event()

        def step_with_gather(i):
            b = i % NB
            stream.wait_event(done[b])  # buffer b's previous gather has read it
            model.process_batch_device(x_dev.data_ptr(), y2[b].data_ptr(), B, n, n, n, stream.cuda_stream)
            ready.record(stream)
            side.wait_event(ready)
            with torch.cuda.stream(side):
                dist.all_gather_into_tensor(gathered[b].view(-1), y2[b].view(-1))
                done[b].record(side)

        # The collective finds its SMs in the last, partly filled round of the persistent kernel (4096 streams over 296 CTAs =
        # 13.8 rounds: 24 SMs idle for the last ~0.7 ms of a step).  Reserving SMs for it outright (nam_b200_set_reserved_sms)
        # was measured and costs a whole extra round (4 SMs: 288 CTAs -> 15 rounds, +8 %), so none are reserved here.
        for i in range(max(args.warmup, NB)):
            step_with_gather(i)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record(stream)
        for i in range(args.steps):
            step_with_gather(i)
        stream.wait_stream(side)
        g1.record(stream)
        barrier()
        t = torch.tensor([g0.elapsed_time(g1)], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        with_ms = float(t.item()) / args.steps
        value_with_gather = world * B * n / (with_ms * 1e-3) / 1e6
        # the collective alone, back to back, for its bus bandwidth
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(5):
            dist.all_gather_into_tensor(gathered[0].view(-1), y2[0].view(-1))
        a1.record()
        torch.cuda.synchronize()
        t = torch.tensor([a0.elapsed_time(a1) / 5], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        gms = float(t.item())
        gather = {"ms_per_step": gms, "bytes_per_rank": int(y_dev.numel() * 4),
                  "busbw_GBs": y_dev.numel() * 4 * (world - 1) / (gms * 1e-3) / 1e9,
                  "step_ms_with_gather_overlapped": with_ms, "step_ms_without": total_ms_max / args.steps,
                  "hidden_fraction": min(1.0, max(0.0, 1.0 - (with_ms - total_ms_max / args.steps) / gms)) if gms > 0 else None,
                  "reserved_sms": 0,
                  "what": "ncclAllGather (torch.distributed all_gather_into_tensor) of each rank's outputs on a side "
                          "stream, overlapped with the next steps' kernels (three output buffers; it runs on the SMs the last, "
                          "partly filled round of the persistent kernel leaves idle); every rank ends up with all N x batch streams"}
        # the gathered block really holds every rank's outputs
        torch.cuda.synchronize()
        assert torch.equal(gathered[(args.steps - 1) % NB][rank], y2[(args.steps - 1) % NB])

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- the other configurations BASELINE.json names, device-resident, a few steps each (N = 1 only) ----
    fp32_packed = nb.measure_fp32_tflops(local_rank, packed=True)
    fp32_scalar = nb.measure_fp32_tflops(local_rank, packed=False)
    fp32_peak = max(fp32_packed, fp32_scalar)  # the roof is the best FP32 FMA rate the SMs can be measured to issue
    secondary = None
    if world == 1 and not args.no_secondary and args.model == MODEL:
        secondary = {}

        def quick(name, model_name, b, frames, steps=8, **kw):
            try:
                m2 = nb.get_dsp(fx.load_model(model_name), batch=b, device=local_rank, fast_tanh=fast, **kw)
                m2.Reset(48000.0, frames)
                xi = torch.from_numpy(fx.synthetic_batch(b, frames, seed=7)).cuda()
                yo = torch.empty_like(xi)
                torch.cuda.synchronize()
                for _ in range(3):
                    m2.process_batch_device(xi.data_ptr(), yo.data_ptr(), b, frames, frames, frames, stream.cuda_stream)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(steps):
                    m2.process_batch_device(xi.data_ptr(), yo.data_ptr(), b, frames, frames, frames, stream.cuda_stream)
                e1.record(stream)
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / steps
                v = b * frames / (ms * 1e-3) / 1e6
                secondary[name] = {"Msamples_per_s": v, "ms_per_step": ms, "streams": b, "frames_per_step": frames,
                                   "rtf_48k_per_stream": v * 1e6 / 48000.0 / b,
                                   "tflops": m2.flops_per_frame * v * 1e6 / 1e12,
                                   "frac_of_fp32_fma_peak": m2.flops_per_frame * v * 1e6 / 1e12 / fp32_peak,
                                   "jit": m2.jit_state}
                m2.close()
            except Exception as exc:  # a secondary workload must never cost the headline line
                secondary[name] = {"error": str(exc)[:200]}

        quick("wavenet_a1_standard_batch1", MODEL, 1, 4096, steps=32)
        quick("wavenet_a1_standard_batch1_wavefront_tiles", MODEL, 1, 4096, steps=32, tile_mode=1)
        quick("wavenet_a1_standard_batch1_one_96000_frame_call", MODEL, 1, 96000, steps=16)
        quick("wavenet_a1_standard_batch1_one_96000_frame_call_tile512", MODEL, 1, 96000, steps=16, kernel_geometry=2)
        quick("wavenet_a1_standard_batch16", MODEL, 16, 4096, steps=16)
        quick("wavenet_a1_standard_batch256", MODEL, 256, 4096)
        quick("wavenet_a1_standard_batch4096_64frame_calls", MODEL, 4096, 64, steps=32)
        quick("wavenet_a1_standard_batch4096_128frame_calls", MODEL, 4096, 128, steps=32)
        quick("a2_full_batch4096", "a2_full", 4096, 4096, steps=4)
        quick("lstm_batch4096", "lstm", 4096, 4096, steps=4)
        # latency roofline of the recurrence (SURVEY.md 8d: streams / step latency).  4096 streams are 512 warps on 592
        # schedulers: every warp issues alone, so the step is bound by its dependent chain.  Chain of the gate-split
        # kernel for a 1-layer cell (instruction latencies of the microarchitecture guide: FFMA / FMUL 4, SHFL ~25, MUFU.RCP
        # ~20): gate FMAs (1 + H + bias) x 4  ->  fast_tanh 45  ->  shuffle 25  ->  cell update 8  ->  fast_tanh 45  ->  h 4.
        if "error" not in secondary["lstm_batch4096"]:
            big = secondary["lstm_batch4096"]
            H = 3
            chain_cycles = (1 + H + 1) * 4 + 45 + 25 + 8 + 45 + 4
            ns_big = big["ms_per_step"] * 1e6 / big["frames_per_step"]
            ns_chain = chain_cycles / 1.965
            big["roofline"] = {"bound": "latency of one recurrence step", "ns_per_step": ns_big,
                               "critical_path_cycles_estimate": chain_cycles, "critical_path_ns_at_1965MHz": ns_chain,
                               "frac": ns_chain / ns_big, "steps_per_s_per_stream": 1e9 / ns_big,
                               "note": "serial in time: throughput = streams in flight / step latency (26 Gsamples/s = 4096 "
                                       "streams / 155 ns); the FLOP fraction is not the bound"}
        quick("wavenet_a2_max_batch4096_general_kernel", "wavenet_a2_max", 4096, 1024, steps=2)

    # ---- roofline of the fused kernel (one launch per step) ----
    peaks = load_peaks()
    kernel_ms = statistics.mean(step_ms)  # one kernel per step on this stream: event-to-event == launch duration
    flops_per_launch = flops_per_frame * B * n
    achieved_tf = flops_per_launch / (kernel_ms * 1e-3) / 1e12
    alg_bytes = B * n * 8.0 + 2.0 * state_bytes * B  # in + out + history read & written once per launch
    roofline = {
        "bound": "fp32_fma",
        "achieved": achieved_tf,
        "peak": fp32_peak,
        "unit": "TFLOP/s",
        "frac": achieved_tf / fp32_peak if fp32_peak > 0 else None,
        "peak_source": "max of the self-measured FP32 FMA issue rates on this GPU (nam_b200_measure_fp32_tflops): "
                       f"scalar FFMA {fp32_scalar:.1f}, packed FFMA2 {fp32_packed:.1f} TFLOP/s; MEASURED_PEAKS.json "
                       "carries no FP32 figure (nominal: 148 SMs x 128 FMA/clk x 1.965 GHz = 74.5)",
        "kernel": ("wavenet_spec_kernel (the model compiled by NVRTC at load: weights as FFMA immediates, history staged by "
                   "cp.async.bulk)" if jit_state == 1 else "wavenet_fused_kernel (precompiled, weights in shared memory)"),
        "jit": {"state": jit_state, "note": jit_note},
        "flops_per_launch": flops_per_launch,
        "kernel_ms": kernel_ms,
        "traffic": None,
        "hbm": {"algorithmic_bytes_per_launch": alg_bytes, "achieved_GBs": alg_bytes / (kernel_ms * 1e-3) / 1e9,
                "peak_GBs": peaks["hbm_gbs"], "frac": alg_bytes / (kernel_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                "of": peaks["_source"]},
        "tensor": {"frac_of_bf16_peak": achieved_tf / peaks["bf16_tflops"], "of": peaks["_source"],
                   "note": "kernel uses the FP32 FMA pipe, not tensor cores (1e-5 parity forbids TF32/BF16 operands)"},
    }
    # DRAM bytes of one launch from the committed ncu --set full capture of this command's default shape
    prof = ROOT / "profiles" / ("r02_traffic.json" if jit_state == 1 else "r01_traffic.json")
    if prof.exists() and args.model == MODEL and (B, n) == (4096, 4096) and args.geometry == 0 and fast:
        try:
            t = json.loads(prof.read_text())
            roofline["traffic"] = t.get("dram_bytes_per_launch_at_bench_shape")
            roofline["traffic_source"] = t.get("source")
        except Exception:
            pass

    cpu = None
    if not args.no_cpu_baseline and world == 1 and rank == 0:  # reported at N = 1 only
        cframes = 96000  # benchmodel's 2 s of audio per stream; ~1 s wall per thread count tried
        arms = cpu_arms(nam, fast, cframes, 4)
        best = arms[arms["kind"]]
        cpu = {"value": best["value"], "unit": "Msamples/s", "cores": best["cores"], "kind": arms["kind"],
               "sample": f"{best['streams']} streams x {cframes} frames in {CPU_BLOCK}-frame process() calls "
                         f"({best['seconds']:.1f} s wall on {best['cores']} threads), {best['flags']}, same tanh regime",
               "port": arms.get("port"), "reference_build": arms.get("reference", arms.get("reference_error"))}
        if secondary is not None and "a2_full_batch4096" in secondary and "error" not in secondary["a2_full_batch4096"]:
            # the A2 bar: the reference serves this shape with its own optimised kernel (A2FastModel,
            # NAM/wavenet/a2_fast.cpp:487-764; protocol of tools/bench_a2_fast.cpp:223-297: 64-frame blocks)
            try:
                a2 = cpu_arms(fx.load_model("a2_full"), fast, 48000, 2)
                b2 = a2[a2["kind"]]
                secondary["a2_full_batch4096"]["cpu_baseline"] = {
                    "value": b2["value"], "unit": "Msamples/s", "cores": b2["cores"], "kind": a2["kind"],
                    "port": a2.get("port"), "reference_build": a2.get("reference", a2.get("reference_error")),
                    "note": "reference build = A2FastModel (NAM_ENABLE_A2_FAST, the default build)"}
            except Exception as exc:
                secondary["a2_full_batch4096"]["cpu_baseline"] = {"error": str(exc)[:200]}

    line = {
        "metric": metric_name(args),
        "value": value,
        "unit": "Msamples/s",
        "n_gpus": world,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": total_ms_max / args.steps,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": workload_config(args),
        "rtf_48k_aggregate": value * 1e6 / 48000.0,
        "rtf_48k_per_stream": value * 1e6 / 48000.0 / (world * B),
        "clocks": clocks.summary(),
        "e2e": e2e,
        "gpu_launches": int(launches),
        "roofline": roofline,
        "cpu_baseline": cpu,
        "secondary": secondary,
    }
    if gather is not None:
        line["value_with_gather"] = value_with_gather
        line["nccl_gather"] = gather
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
