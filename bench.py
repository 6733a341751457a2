#!/usr/bin/env python
"""Benchmark of the RAFT inference hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA backend
    python bench.py --impl reference --steps K --warmup W    # the reference algorithm on the host CPU

metric  : frame-pairs/sec, RAFT, 1024x436, 12 refinement iterations, f16 storage, batch 8 per GPU
          (BASELINE.json configs[1]); weak scaling over N GPUs (frame pairs shard, no collective on
          the data path -- SURVEY.md section 8(e)).
value   : whole-job pairs/s with inputs already resident in HBM (CUDA events, max over ranks).
e2e     : the same through the public API with HOST (pinned) inputs: every step's frames are copied H2D and
          every step's predicted flow D2H inside the timed region (copies ride a side stream and overlap the
          neighbouring step's compute, as a real frame pipeline would).
roofline: for the kernel class that dominates the step, algorithmic FLOPs (or bytes) per launch over
          its live CUDA-event duration (a separate instrumented pass of the same workload), against
          MEASURED_PEAKS.json.  `kernels` lists every class, incl. the corr-lookup HBM GB/s.
cpu_baseline / --impl reference: oracle/raft_oracle.py (torch-fp32 port of the reference algorithm,
          pinned to reference-generated vectors) on the box's host cores, bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

T_START = time.time()


def log(msg: str) -> None:
    """Progress on stderr (the JSON result line is the only thing written to stdout)."""
    print(f"[bench +{time.time() - T_START:6.1f}s] {msg}", file=sys.stderr, flush=True)


def host_cores() -> int:
    """Cores this process may really use: min(cpu_count, affinity mask, cgroup cpu.max quota)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except (OSError, ValueError):
        pass
    return max(1, n)


FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="raft")
    ap.add_argument("--batch", type=int, default=8, help="frame pairs per GPU per step")
    ap.add_argument("--height", type=int, default=436)
    ap.add_argument("--width", type=int, default=1024)
    ap.add_argument("--iters", type=int, default=12)
    ap.add_argument("--dtype", default="fp16", choices=["fp16", "bf16", "fp32"])
    ap.add_argument("--kernel-impl", type=int, default=0, help="0 auto, 1 SIMT, 2 tcgen05")
    ap.add_argument("--inflight", type=int, default=1, help="frame-pair batches in flight per GPU (ptlflow_b200.pipeline.FramePipeline); 1 = one stream")
    ap.add_argument("--cuda-graph", type=int, default=1, help="1: one CUDA graph launch per forward (default); 0: eager launches")
    ap.add_argument("--fp32-context", action="store_true", help="accuracy mode: context encoder in fp32 (RAFT.enable_fp32_context)")
    ap.add_argument("--protocol-samples", type=int, default=12, help="synchronised single forwards for the model_benchmark.py protocol (0 = skip)")
    ap.add_argument("--sustained-seconds", type=float, default=5.0, help="length of the sustained loop (0 = skip)")
    ap.add_argument("--alternate-corr", action="store_true", help="on-the-fly correlation (no 4D volume), BASELINE config 4")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-comparators", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-baseline-seconds", type=float, default=12.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy, float32 (float64 stays float64), "
                    "at most 64 MB in all (see dump_outputs)")
    return ap.parse_args()


DUMP_BUDGET_BYTES = 64_000_000


def host_outputs(out) -> dict:
    """The tensors of a forward's output dict as host numpy arrays: float64 stays float64, everything else becomes float32."""
    import numpy as np

    return {k: v.detach().cpu().numpy().astype(np.float64 if v.dtype == torch.float64 else np.float32)
            for k, v in out.items() if isinstance(v, torch.Tensor)}


def dump_outputs(arrays: dict, directory: str) -> None:
    """Write each array as ``<name>.npy`` so that two builds can be compared output for output.  When the arrays exceed
    DUMP_BUDGET_BYTES together, each is cut to the same share of its elements: a fixed-seed sample of flat positions, in
    order, so the same arguments always select the same positions."""
    import numpy as np

    os.makedirs(directory, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    for name, a in sorted(arrays.items()):
        if total > DUMP_BUDGET_BYTES:
            flat = a.reshape(-1)
            keep = np.sort(np.random.default_rng(0).choice(flat.size, flat.size * DUMP_BUDGET_BYTES // total, replace=False))
            a = flat[keep]
        np.save(os.path.join(directory, name + ".npy"), a)
    log(f"outputs of the last timed step written to {directory}: {', '.join(sorted(arrays))}")


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        p["_source"] = "measured (MEASURED_PEAKS.json)"
        return p
    p = dict(FALLBACK_PEAKS)
    p["_source"] = "fallback (B200_PROFILING.md)"
    return p


# ----------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.lines, self.proc = [], None
        try:
            uuid = str(torch.cuda.get_device_properties(device_index).uuid)
            sel = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
        except Exception:
            sel = str(device_index)
        self.cmd = ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100", "-i", sel]

    def start(self):
        try:
            # On a fresh box the first nvidia-smi of the boot takes seconds to attach to the driver and stalls the
            # launching threads of a running CUDA process while it does: pay that once, synchronously, before anything
            # is timed (measured: 23 ms/step instead of 9 when its start-up overlapped the timed loop).
            subprocess.run(["nvidia-smi", "-L"], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, timeout=120)
            self.proc = subprocess.Popen(self.cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except (OSError, subprocess.TimeoutExpired):
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def wait_first_sample(self, timeout_s: float = 60.0):
        """nvidia-smi's start-up (driver / NVML attach) stalls the launching threads of a running CUDA process for
        tens of milliseconds: let it finish before anything is timed."""
        t0 = time.perf_counter()
        while self.proc is not None and not self.lines and time.perf_counter() - t0 < timeout_s:
            time.sleep(0.05)

    def mark(self):
        """Samples before this point (warm-up) are dropped: the clocks line describes the timed region only."""
        self.lines = []

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); smax.append(float(parts[1])); power.append(float(parts[2]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(smax), "power_w_max": max(power), "samples": len(sm),
                "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------
# algorithmic work of one step (DESIGN.md "roofline arithmetic")
# ----------------------------------------------------------------------------------------------
def algorithmic_work(model, B, H8, W8, iters, esize):
    """FLOPs / bytes per step for each kernel class, from the layer shapes the engine packed."""
    from ptlflow_b200 import _lib

    eng = model._engine
    P = B * H8 * W8
    per_iter, once, exe_iter, exe_once = 0, 0, 0, 0
    ref_layers = (_lib.L_CONVC1, _lib.L_CONVC2, _lib.L_CONVF2, _lib.L_CONV, _lib.L_GRU_ZR1, _lib.L_GRU_Q1, _lib.L_GRU_ZR2, _lib.L_GRU_Q2,
                  _lib.L_FLOW1, _lib.L_FLOW2, _lib.L_MASK1, _lib.L_MASK2, _lib.L_AGG_V)
    if eng.layers[_lib.L_CONVF1].weight_k is None:
        ref_layers += (_lib.L_CONVF1,)  # (on tcgen05 convf1 runs in its own kernel class, "flowconv")
    for lid in ref_layers:  # the reference's layers (update.py:94-153): the ALGORITHMIC work
        pk = eng.layers.get(lid)
        if pk is None:
            continue
        fl = 2 * pk.Cin * pk.KH * pk.KW * pk.Cout * P
        if lid in (_lib.L_MASK1, _lib.L_MASK2):
            once += fl
        else:
            per_iter += fl
    # what the tensor-core path EXECUTES: the context third of the GRU convolutions once per forward, convc2 | convf2 as one
    # block-diagonal layer (zeros included), the flow head's last layer as 18 tap products
    tensor = _lib.L_GRUX_ZR1 in eng.layers
    for lid, pk in eng.layers.items():
        fl = 2 * pk.Cin * pk.KH * pk.KW * pk.Cout * P
        if tensor and lid in (_lib.L_GRU_ZR1, _lib.L_GRU_Q1, _lib.L_GRU_ZR2, _lib.L_GRU_Q2, _lib.L_FLOW2):
            continue
        if _lib.L_CONVC2F2 in eng.layers and lid in (_lib.L_CONVC2, _lib.L_CONVF2):
            continue
        if lid == _lib.L_CONVF1 and pk.weight_k is not None:
            continue
        if lid in (_lib.L_MASK1, _lib.L_MASK2, _lib.L_CTX_ZR1, _lib.L_CTX_Q1, _lib.L_CTX_ZR2, _lib.L_CTX_Q2):
            exe_once += fl
        else:
            exe_iter += fl
    L, r = model.corr_levels, model.corr_radius
    planes = L * (2 * r + 1) ** 2
    lookup_bytes = iters * P * (L * (2 * r + 2) ** 2 * esize + planes * esize + 8)
    N = H8 * W8
    C = model.fnet.conv2.out_channels
    vol_elems = sum((H8 >> l) * (W8 >> l) for l in range(L))
    return {
        "conv": {"flops": per_iter * iters + once, "executed_flops": exe_iter * iters + exe_once},
        "lookup": {"bytes": lookup_bytes},
        # a1 + a2 in one launch: both feature maps read once, every pyramid level written once (SURVEY.md section 8(d))
        "volume": {"bytes": B * (2 * N * C * esize + N * vol_elems * esize), "flops": 2 * B * N * N * C},
        "pool": {"bytes": B * N * esize * (vol_elems - H8 * W8 + sum((H8 >> l) * (W8 >> l) for l in range(L - 1)))},
        "upsample": {"bytes": P * (576 * esize + 8) + B * 2 * 64 * N * 4},
    }


KC_NAMES = ["volume", "pool", "lookup", "onthefly", "conv", "upsample", "misc", "enc_affine", "enc_stats", "enc_conv1", "flowconv", "gather"]


def run_ours(args):
    import ctypes as C
    from argparse import Namespace

    import ptlflow_b200 as pb
    from ptlflow_b200 import _lib, sharding

    rank, local_rank, world = sharding.env_rank_world()
    assert world == max(1, args.gpus) or world == 1, f"WORLD_SIZE={world} but --gpus {args.gpus}"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # NCCL may print its version banner on stdout (NCCL_DEBUG=VERSION on some boxes); stdout carries exactly one JSON line,
    # so file descriptor 1 points at stderr while the process group comes up and the first collective runs
    sys.stdout.flush()
    saved_fd = os.dup(1)
    os.dup2(2, 1)
    try:
        sharding.init_process_group("nccl")
        sharding.barrier()
        torch.cuda.synchronize()
    finally:
        sys.stdout.flush()
        os.dup2(saved_fd, 1)
        os.close(saved_fd)
    lib = _lib.load()

    dtype = {"fp16": torch.float16, "bf16": torch.bfloat16, "fp32": torch.float32}[args.dtype]
    torch.manual_seed(1234)
    mkw = dict(iters=args.iters)
    if args.alternate_corr:
        mkw["alternate_corr"] = True
    model = pb.get_model(args.model, args=Namespace(model=Namespace(**mkw)))
    sd_fp32 = {k: v.detach().clone() for k, v in model.state_dict().items()}  # the fp32 weights the reference would hold
    if args.fp32_context:
        model.enable_fp32_context()
    model = model.eval().to(dev).to(dtype)
    model.kernel_impl = args.kernel_impl
    model.use_cuda_graph = bool(args.cuda_graph)

    B, H, W = args.batch, args.height, args.width
    pool = 3
    g = torch.Generator().manual_seed(100 + rank)
    host = [torch.rand(B, 2, 3, H, W, generator=g).to(dtype).pin_memory() for _ in range(pool)]
    devin = [h.to(dev) for h in host]
    host_out = torch.empty((B, 1, 2, H, W), dtype=dtype).pin_memory()

    def launches_now():
        return int(lib.pfb_launch_count(-1)) + int(model.graph_launches_replayed)

    def step_resident(i):
        return model({"images": devin[i % pool]})

    # e2e: what a caller feeding frames from host memory runs.  Two device input slots; the H2D copy of step i+1 and the
    # D2H copy of step i's flow ride a side stream while step i / i+1 computes (PCIe is full duplex).  Every step's input
    # really comes from pinned host memory and every step's flow really lands in pinned host memory inside the timed region.
    copy_stream = torch.cuda.Stream(device=dev)
    dev_in = [torch.empty_like(devin[0]) for _ in range(2)]
    h2d_done = [torch.cuda.Event() for _ in range(2)]
    slot_free = [torch.cuda.Event() for _ in range(2)]

    def issue_h2d(i):
        slot = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(slot_free[slot])
            dev_in[slot].copy_(host[i % pool], non_blocking=True)
            h2d_done[slot].record(copy_stream)

    def run_e2e(n):
        main = torch.cuda.current_stream(dev)
        for sl in range(2):
            slot_free[sl].record(main)
        issue_h2d(0)
        for i in range(n):
            if i + 1 < n:
                issue_h2d(i + 1)
            slot = i % 2
            main.wait_event(h2d_done[slot])
            out = model({"images": dev_in[slot]})
            slot_free[slot].record(main)
            flows = out["flows"]
            done = torch.cuda.Event()
            done.record(main)
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(done)
                host_out.copy_(flows, non_blocking=True)
            flows.record_stream(copy_stream)
        main.wait_stream(copy_stream)

    # --inflight > 1: several batches in flight (ptlflow_b200.pipeline.FramePipeline: one stream + host thread + CUDA graph
    # per slot).  Default 1: one stream, one graph launch per forward -- the protocol of SURVEY.md section 8(d).
    pipe = None
    if args.inflight > 1:
        from ptlflow_b200.pipeline import FramePipeline

        pipe = FramePipeline(model, depth=args.inflight, device=dev)
        host_outs = [torch.empty((B, 1, 2, H, W), dtype=dtype).pin_memory() for _ in range(args.inflight)]

    last = {}  # the most recent run_value's last step: its outputs (or, in flight, its pending result) for --dump-outputs

    def run_value(n):
        if pipe is None:
            for i in range(n):
                last["out"] = step_resident(i)
        else:
            res = [pipe.submit({"images": devin[i % pool]}) for i in range(n)]
            pipe.drain()
            for r in res:
                r.enqueued()  # re-raises what a slot thread caught: a failed forward must not count as a fast one
            last["out"] = res[-1]

    def run_e2e_any(n):
        if pipe is None:
            run_e2e(n)
        else:
            # pinned host frames in, predicted flow back to pinned host memory, every step
            res = [pipe.submit({"images": host[i % pool]}, host_out=host_outs[i % args.inflight]) for i in range(n)]
            pipe.drain()
            for r in res:
                r.enqueued()

    log(f"model on {dev}, {args.dtype}, batch {B}, {args.inflight} batch(es) in flight, cuda graph {'on' if model.use_cuda_graph else 'off'}; warming up")
    sampler = ClockSampler(local_rank)
    sampler.start()
    with torch.no_grad():
        for i in range(max(3, args.warmup)):
            step_resident(i)
            torch.cuda.synchronize()
            log(f"warm-up step {i} done")
        if pipe is not None:  # the slots' threads tune cuDNN (thread-local cache), capture their graphs and allocate their scratch
            run_value(max(3, args.warmup) * args.inflight)
            run_e2e_any(args.inflight)
            torch.cuda.synchronize()
            log("pipeline warm-up done")
        run_e2e_any(2)
        torch.cuda.synchronize()

        sampler.wait_first_sample()
        time.sleep(0.5)
        run_value(args.steps)  # pre-roll: an untimed copy of the timed loop right before it
        torch.cuda.synchronize()
        sampler.mark()

        def timed(fn, n):
            sharding.barrier(); torch.cuda.synchronize()
            n0 = launches_now()
            t0 = time.perf_counter()
            v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            v0.record()
            fn(n)
            v1.record()
            torch.cuda.synchronize()
            wall_ms = (time.perf_counter() - t0) * 1e3
            sharding.barrier()
            return sharding.max_over_ranks(max(v0.elapsed_time(v1), 0.0), dev), sharding.max_over_ranks(wall_ms, dev), launches_now() - n0

        # ---- value: device-resident inputs, exactly K steps ----
        ms_value, _, launches = timed(run_value, args.steps)
        log(f"resident: {ms_value / args.steps:.3f} ms/step")
        # ---- e2e: pinned host inputs, H2D + forward + D2H of the flow every step ----
        ms_e2e_ev, ms_e2e_wall, _ = timed(run_e2e_any, args.steps)
        ms_e2e = max(ms_e2e_ev, ms_e2e_wall)
        e2e_remeasured = False
        if ms_e2e > 1.25 * ms_value:
            # the end-to-end loop adds two PCIe copies per step that overlap the compute; a reading this far above the resident
            # loop caught a host-side transient (seen on shared boxes: 561 vs 919 pairs/s on consecutive runs) -- measured once more
            ms2_ev, ms2_wall, _ = timed(run_e2e_any, args.steps)
            ms_e2e = min(ms_e2e, max(ms2_ev, ms2_wall))
            e2e_remeasured = True
        value_remeasured = False
        if ms_value > 1.25 * ms_e2e:  # the resident loop does strictly less work: a slower reading caught a transient
            ms_value, _, launches = timed(run_value, args.steps)
            value_remeasured = True
            log(f"resident (re-measured): {ms_value / args.steps:.3f} ms/step")
        dumped = None
        if args.dump_outputs and rank == 0:
            # taken before any later loop calls run_value again: the last timed step always reads devin[(steps - 1) % pool]
            out = last.pop("out")
            dumped = host_outputs(out if pipe is None else out.get())
        clocks = sampler.stop()
        log(f"e2e: {ms_e2e / args.steps:.3f} ms/step; clocks {clocks}")

        # ---- protocol of the reference's model_benchmark.py:421-466 (SURVEY.md section 8(d)): fresh torch.rand per sample
        # (made on the CPU, moved and converted OUTSIDE the timed region), synchronise before and after every single
        # forward, first forward dropped, median ----
        proto = None
        if args.protocol_samples > 0:
            times = []
            gp = torch.Generator().manual_seed(555 + rank)
            for i in range(args.protocol_samples + 1):
                x = torch.rand(B, 2, 3, H, W, generator=gp).to(dev).to(dtype)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                model({"images": x})
                torch.cuda.synchronize()
                if i > 0:
                    times.append((time.perf_counter() - t0) * 1e3)
            med = statistics.median(times)
            med = sharding.max_over_ranks(med, dev)
            proto = {"what": "median wall time of synchronised single forwards on fresh torch.rand frames (model_benchmark.py:421-466), one stream",
                     "samples": len(times), "median_ms": round(med, 4), "min_ms": round(min(times), 4), "max_ms": round(max(times), 4),
                     "value": round(B * world / (med * 1e-3), 2), "unit": "pairs/s"}
            log(f"protocol: median {med:.3f} ms per synchronised forward")

        # ---- sustained: the resident loop for >= N seconds (the K-step number above is a burst of ~0.1 s) ----
        sustained = None
        if args.sustained_seconds > 0:
            per = max(1e-3, ms_value / args.steps)
            n_sus = max(args.steps, int(args.sustained_seconds * 1e3 / per) + 1)
            s2 = ClockSampler(local_rank)
            s2.start(); s2.wait_first_sample(); s2.mark()
            ms_sus, _, _ = timed(run_value, n_sus)
            c2 = s2.stop()
            sustained = {"seconds": round(ms_sus * 1e-3, 2), "steps": n_sus, "ms_per_step": round(ms_sus / n_sus, 4),
                         "value": round(B * n_sus * world / (ms_sus * 1e-3), 2), "unit": "pairs/s", "clocks": c2}
            log(f"sustained: {ms_sus / n_sus:.3f} ms/step over {ms_sus * 1e-3:.1f} s")

        # ---- strong scaling beside weak (SURVEY.md section 8(d)): the SAME 8 pairs split over the ranks ----
        strong = None
        if world > 1 and B % world == 0:
            bs = B // world
            sub = [d[:bs].contiguous() for d in devin]
            for i in range(3):
                model({"images": sub[i % pool]})
            ms_st, _, _ = timed(lambda n: [model({"images": sub[i % pool]}) for i in range(n)], args.steps)
            strong = {"total_pairs_per_step": B, "pairs_per_step_per_gpu": bs, "ms_per_step": round(ms_st / args.steps, 4),
                      "value": round(B * args.steps / (ms_st * 1e-3), 2), "unit": "pairs/s"}

        # ---- output check (outside every timed region): this run's flow against the fp32 oracle on the same frames ----
        parity = None
        if rank == 0 and not args.no_parity:
            parity = parity_check(args, model, sd_fp32, devin[0], dev)
            log(f"parity: {parity}")

        # ---- instrumented pass: live per-kernel-class durations, eager launches (not part of the numbers above) ----
        prof_steps = 2
        was_graph = model.use_cuda_graph
        model.use_cuda_graph = False
        # one stream, no fork / join: a kernel's span must not contain a kernel of another class running beside it
        was_fork = (getattr(model, "fork_flow", False), getattr(model, "fork_encoders", False))
        model.fork_flow = model.fork_encoders = False
        step_resident(0)
        torch.cuda.synchronize()
        lib.pfb_profile_enable(1)
        t_ev0, t_ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_ev0.record()
        for i in range(prof_steps):
            step_resident(i)
        t_ev1.record()
        ms_arr, n_arr = (C.c_double * 16)(), (C.c_ulonglong * 16)()
        _lib.check(lib.pfb_profile_collect(ms_arr, n_arr, 16), "profile_collect")
        lib.pfb_profile_enable(0)
        ms_prof_step = t_ev0.elapsed_time(t_ev1) / prof_steps
        model.use_cuda_graph = was_graph
        model.fork_flow, model.fork_encoders = was_fork
        log("instrumented pass done")
        if pipe is not None:
            pipe.close()

        comparators = None
        if rank == 0 and world == 1 and not args.no_comparators:
            comparators = same_gpu_comparators(args, dev)
            log(f"same-GPU comparators: {comparators}")

    H8, W8 = (H + 7) // 8, (W + 7) // 8
    esize = 4 if dtype == torch.float32 else 2
    work = algorithmic_work(model, B, H8, W8, args.iters, esize)
    peaks = load_peaks()
    kernels = {}
    ours_ms = 0.0
    for kc, name in enumerate(KC_NAMES):
        if n_arr[kc] == 0:
            continue
        ms_step = ms_arr[kc] / prof_steps
        ours_ms += ms_step
        ent = {"ms_per_step": round(ms_step, 4), "launches_per_step": int(n_arr[kc] // prof_steps)}
        w = work.get(name, {})
        if "flops" in w and name == "conv":
            ent["tflops"] = round(w["flops"] / (ms_step * 1e-3) / 1e12, 2)
            ent["frac_of_bf16_burst_peak"] = round(ent["tflops"] / peaks["bf16_tflops"], 4)
            ent["frac_of_bf16_sustained_peak"] = round(ent["tflops"] / peaks["bf16_tflops_sustained"], 4)
            ent["executed_tflops"] = round(w["executed_flops"] / (ms_step * 1e-3) / 1e12, 2)
            ent["note"] = "tflops = the reference layers' FLOPs (update.py:94-153) over the measured time; executed_tflops = what the kernels issue (context third of the GRU once per forward, block-diagonal convc2|convf2)"
        if "bytes" in w:
            ent["algorithmic_gbs"] = round(w["bytes"] / (ms_step * 1e-3) / 1e9, 1)
            ent["frac_of_hbm_peak"] = round(ent["algorithmic_gbs"] / peaks["hbm_gbs"], 4)
        kernels[name] = ent
    kernels["_not_this_library"] = {"ms_per_step": round(max(0.0, ms_prof_step - ours_ms), 4),
                                    "what": "cuDNN encoder convolutions + torch glue: instrumented step time minus this library's classes"}
    cand = {k: v for k, v in kernels.items() if not k.startswith("_")}
    dominant = max(cand, key=lambda k: cand[k]["ms_per_step"]) if cand else None
    roofline = None
    if dominant == "conv":
        e = kernels["conv"]
        traffic = None  # DRAM bytes per launch from the committed ncu --set full capture of the same command
        for tname in ("r02_conv_umma_traffic.json", "r01_conv_umma_traffic.json"):
            tpath = os.path.join(ROOT, "profiles", tname)
            if os.path.exists(tpath):
                with open(tpath) as f:
                    traffic = round(json.load(f)["dram_bytes_per_launch"])
                break
        # the timed region is a burst (~0.1 s at ~1.9 GHz), so the burst bf16 peak is the matching denominator
        roofline = {"kernel": "update-block conv (implicit GEMM, tcgen05)", "bound": "tensor", "achieved": e["tflops"],
                    "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": e["frac_of_bf16_burst_peak"],
                    "frac_of_sustained_peak": e["frac_of_bf16_sustained_peak"],
                    "traffic": traffic, "peak_source": peaks["_source"] + ", burst bf16 GEMM",
                    "algorithmic_flops_per_launch": round(work["conv"]["flops"] / max(1, e["launches_per_step"]))}
    elif dominant is not None and "algorithmic_gbs" in kernels[dominant]:
        e = kernels[dominant]
        roofline = {"kernel": dominant, "bound": "hbm", "achieved": e["algorithmic_gbs"], "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": e["frac_of_hbm_peak"], "traffic": None, "peak_source": peaks["_source"]}
    # north_star's headline fraction: correlation volume build + all lookups against the HBM roofline
    corr_frac = None
    if "volume" in kernels and "lookup" in kernels:
        t_corr = (kernels["volume"]["ms_per_step"] + kernels["lookup"]["ms_per_step"]) * 1e-3
        bytes_corr = work["volume"]["bytes"] + work["lookup"]["bytes"]
        corr_frac = {"algorithmic_bytes_per_step": int(bytes_corr), "ms_per_step": round(t_corr * 1e3, 4),
                     "achieved_gbs": round(bytes_corr / t_corr / 1e9, 1), "frac_of_hbm_peak": round(bytes_corr / t_corr / 1e9 / peaks["hbm_gbs"], 4)}

    pairs = B * args.steps * world
    value = pairs / (ms_value * 1e-3)
    e2e_value = pairs / (ms_e2e * 1e-3)
    result = {
        "metric": "frame-pairs/sec RAFT 1024x436 12-iter",
        "value": round(value, 3), "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": round(ms_value / args.steps, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": {"fp16": "f16", "bf16": "bf16", "fp32": "f32"}[args.dtype] + " storage, f32 accumulate/coordinates",
        "data": "synthetic (torch.rand frames, random-init weights, seed 1234)",
        "config": {"workload": f"{args.model} {W}x{H} {args.iters} iters, batch {B} per GPU (BASELINE.json configs[1])",
                   "pairs_per_step_per_gpu": B, "batches_in_flight_per_gpu": args.inflight, "stream_forks": {"flow_branch": bool(getattr(model, "fork_flow", False)), "encoders": bool(getattr(model, "fork_encoders", False))}, "cuda_graph": bool(model.use_cuda_graph), "alternate_corr": bool(args.alternate_corr),
                   "fp32_context": bool(args.fp32_context), "value_remeasured": value_remeasured, "e2e_remeasured": e2e_remeasured,
                   "parallelism": f"replicas x{world}, frame pairs sharded, no data-path collective",
                   "l2": "per-step working set (>= 1 GB correlation pyramid at batch 8) exceeds the 126 MB L2; inputs rotate over a pool of 3 batches",
                   "kernel_impl": args.kernel_impl},
        "e2e": {"value": round(e2e_value, 3), "unit": "pairs/s", "ms_per_step": round(ms_e2e / args.steps, 4),
                "h2d_bytes_per_step": int(host[0].numel() * host[0].element_size()),
                "d2h_bytes_per_step": int(host_out.numel() * host_out.element_size())},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "corr_hbm_roofline": corr_frac,
        "protocol": proto,
        "sustained": sustained,
        "strong_scaling": strong,
        "parity": parity,
        "kernels": kernels,
        "same_gpu_comparators": comparators,
    }
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        result["cpu_baseline"] = cpu_baseline(args, args.cpu_baseline_seconds)
    if dumped is not None:
        dump_outputs(dumped, args.dump_outputs)
    if rank == 0:
        print(json.dumps(result), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


def parity_check(args, model, sd_fp32, frames, dev):
    """One forward of the benchmarked model object on (a 2-pair subset of) the benchmarked frames against the fp32 oracle
    run on the same GPU with the model's ORIGINAL fp32 weights (before ``.half()``).  Outside every timed region."""
    from oracle import raft_oracle as O

    n = min(2, frames.shape[0])
    x = frames[:n].contiguous()
    sd = {k: v.to(dev) for k, v in sd_fp32.items()}
    with torch.no_grad(), O.fp32_strict():
        ref = O.raft_forward(sd, x.float(), args.model, iters=args.iters)["flows"]
        out = model({"images": x})["flows_fp32"].float()
    d = (out - ref).abs()
    return {"max_abs_px": round(d.max().item(), 5), "mean_abs_px": round(d.mean().item(), 6), "max_flow_px": round(ref.abs().max().item(), 3),
            "pairs": n, "against": "oracle/raft_oracle.py in fp32 (TF32 off) on the same GPU, holding the model's fp32 weights from before .half()"}


def same_gpu_comparators(args, dev):
    """The reference's algorithm as plain PyTorch-CUDA ops (the oracle port) on the same B200, same workload, timed with the
    model_benchmark.py protocol: fp32 with TF32 off, and half precision like ``model.half()``.  Reported baselines."""
    from oracle import raft_oracle as O
    from oracle import synth

    out = {}
    sd32 = {k: v.to(dev) for k, v in synth.synth_state_dict(O.state_dict_shapes(args.model), 1234).items()}
    B = args.batch
    for name, half in (("pytorch_cuda_fp32_tf32_off", False), ("pytorch_cuda_half", True)):
        try:
            sd = {k: (v.half() if (half and v.is_floating_point()) else v) for k, v in sd32.items()}
            fwd = _half_forward if half else O.raft_forward
            times = []
            for i in range(4):
                x = torch.rand(B, 2, 3, args.height, args.width).to(dev)
                x = x.half() if half else x
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                with torch.no_grad():
                    if half:
                        fwd(sd, x, args.model, args.iters)
                    else:
                        with O.fp32_strict():
                            fwd(sd, x, args.model, iters=args.iters)
                torch.cuda.synchronize()
                if i > 0:
                    times.append((time.perf_counter() - t0) * 1e3)
            med = statistics.median(times)
            out[name] = {"median_ms": round(med, 3), "value": round(B / (med * 1e-3), 2), "unit": "pairs/s", "samples": len(times),
                         "kind": "port (oracle/raft_oracle.py ops on CUDA tensors)", "batch": B}
        except Exception as e:  # noqa: BLE001 -- a comparator must never take the bench line down
            out[name] = {"error": f"{type(e).__name__}: {e}"[:200]}
        torch.cuda.empty_cache()
    return out


def _half_forward(sd, images, variant, iters):
    """raft_forward with every tensor in half precision (what ``model.half()`` does to the reference): the oracle casts to
    fp32 internally, so this wrapper re-implements the cast policy by monkey-free means: run the same functions on half tensors."""
    from oracle import raft_oracle as O

    small, hdim, cdim, _f, cnorm, radius = O.VARIANTS[variant]
    x, pads = O.preprocess(images)
    img1, img2 = x[:, 0], x[:, 1]
    b = img1.shape[0]
    fmaps = O.encoder(torch.cat([img1, img2], 0), sd, "fnet.", "instance", small)
    fmap1, fmap2 = fmaps[:b], fmaps[b:]
    cnet = O.encoder(img1, sd, "cnet.", cnorm, small)
    net, inp = torch.tanh(cnet[:, :hdim]), torch.relu(cnet[:, hdim:hdim + cdim])
    pyr = O.corr_pyramid(O.corr_volume(fmap1, fmap2), 4)
    h8, w8 = fmap1.shape[-2:]
    coords0 = O.coords_grid(b, h8, w8, dtype=images.dtype, device=images.device)
    coords1 = coords0.clone()
    block = O.small_update_block if small else O.basic_update_block
    mask = None
    for _ in range(iters):
        corr = O.corr_lookup(pyr, coords1, radius)
        net, mask, delta = block(net, inp, corr, coords1 - coords0, sd)
        coords1 = coords1 + delta
    flow_small = coords1 - coords0
    up = O.upflow8(flow_small) if mask is None else O.convex_upsample(flow_small, mask)
    return O.unpad(up, pads)


# ----------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference algorithm on the host cores
# ----------------------------------------------------------------------------------------------
def _cpu_setup(args):
    from oracle import raft_oracle as O
    from oracle import synth

    cores = host_cores()
    torch.set_num_threads(cores)
    log(f"cpu arm: {cores} host threads (os.cpu_count()={os.cpu_count()})")
    sd = synth.synth_state_dict(O.state_dict_shapes(args.model), 1234)
    g = torch.Generator().manual_seed(7)

    def one_pair():
        img = torch.rand(1, 2, 3, args.height, args.width, generator=g)
        with torch.no_grad():
            return O.raft_forward(sd, img, args.model, iters=args.iters)

    return one_pair, cores


def cpu_baseline(args, budget_s: float):
    one_pair, cores = _cpu_setup(args)
    t0 = time.perf_counter()
    one_pair()  # warm-up (counted only if it alone exhausts the budget)
    n, dt = 1, time.perf_counter() - t0
    log(f"cpu baseline warm-up pair took {dt:.2f}s")
    if dt < budget_s:
        n, t0 = 0, time.perf_counter()
        while True:
            one_pair(); n += 1
            dt = time.perf_counter() - t0
            if dt >= budget_s or n >= 16:
                break
    return {"value": round(n / dt, 4), "unit": "pairs/s", "cores": cores, "kind": "port",
            "sample": f"{n} single frame pairs of the same workload ({args.model} {args.width}x{args.height}, {args.iters} iters, fp32, batch 1), oracle/raft_oracle.py on torch CPU"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # rank 0 alone runs the CPU arm
    one_pair, cores = _cpu_setup(args)
    for _ in range(max(1, args.warmup)):
        one_pair()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = one_pair()
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(host_outputs(out), args.dump_outputs)
    value = args.steps / dt
    sample = f"each step = 1 frame pair (of the batch of {args.batch}) at {args.width}x{args.height}, {args.iters} iters, fp32"
    print(json.dumps({
        "impl": "reference", "metric": "frame-pairs/sec RAFT 1024x436 12-iter", "value": round(value, 4), "unit": "pairs/s",
        "n_gpus": max(1, args.gpus), "steps": args.steps, "warmup": max(1, args.warmup), "ms_per_step": round(dt / args.steps * 1e3, 2),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic (torch.rand frames, synthetic weights)",
        "config": {"workload": f"{args.model} {args.width}x{args.height} {args.iters} iters, batch {args.batch} per GPU (BASELINE.json configs[1])",
                   "sample": sample},
        "cpu_baseline": {"value": round(value, 4), "unit": "pairs/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": round(value, 4), "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), flush=True)


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
