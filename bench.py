#!/usr/bin/env python
"""bench.py -- env-steps/s of the batched step() hot path (BASELINE.json metric).

    python bench.py --gpus 1 --steps K --warmup W              # our arm (default)
    python bench.py --impl reference --gpus 1 --steps K --warmup W
    torchrun ... bench.py --gpus N ...                          # one rank per GPU
    python bench.py ... --dump-outputs DIR     # + the last timed step's outputs as DIR/*.npy

A "step" is one sync step of one batch: every env of the pool advances once.  Workload at
N=1: BASELINE.json configs[1], CartPole-v1 with num_envs=65536 on one B200.  N>1 is weak
scaling: 65536 envs per GPU, env ids sharded by rank, and -- the path north_star names --
after every step every GPU holds the output columns of ALL envs: `value` at N>1 is measured
WITH that exchange (the engine's own NVLink peer exchange, csrc/exchange.cuh); the
collective-free figure (independent replicas) is reported beside it under `replicas`, the
NCCL all-gather of the same columns under `with_allgather_nccl`.  `value` is measured with
actions and outputs resident in HBM (device-resident C-ABI path, one kernel launch per step,
replayed from a CUDA graph, timestamps taken inside the graph); `e2e` is the same metric
through the reference-facing API (envpool_b200.make(...).step(numpy)) with host buffers,
H2D/D2H inside the timed region.  `configs` carries one line per remaining BASELINE.json
config (3, 4, 5) at the --gpus given.  Rank 0 prints ONE JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# task id -> (engine task, registered max_episode_steps, iopt, #discrete actions or None)
TASKS = {
    "CartPole-v1": ("CartPole", 500, -1, 2),
    "Pendulum-v1": ("Pendulum", 200, 1, None),
    "Acrobot-v1": ("Acrobot", 500, -1, 3),
    "MountainCar-v0": ("MountainCar", 200, -1, 3),
    "FrozenLake-v1": ("FrozenLake", 100, 4, 4),
    "Catch-v0": ("Catch", -1, -1, 3),
    "Taxi-v3": ("Taxi", 200, -1, 6),
    "HalfCheetah-v4": ("HalfCheetah", 1000, -1, None),
}
METRIC = "env steps/sec (whole box)"
L2_BYTES = 126 * 1024 * 1024
MAX_CHAIN = 4096          # steps per captured chain (2-4 kernel nodes each)
DUMP_BYTES = 60 << 20     # --dump-outputs: .npy data under 64 MB, headers included
# fp64 operations per HalfCheetah env step (5 mj_step), from the instruction counts of one
# ncu capture of hc_thread_kernel (profiles/README.md): DFMA = 2, DADD / DMUL = 1
HC_FLOP_PER_ENV_STEP = None


def bench_config(task, n, world, precision):
    """`config` of the JSON line: the SAME dict in both arms (the driver compares them)."""
    tag = " (BASELINE.json configs[1])" if (task, n) == ("CartPole-v1", 65536) else ""
    return {
        "workload": f"{task} sync num_envs={n} per GPU x {world} GPU{tag}",
        "precision": precision, "seed": 0,
        "l2": "GPU arm: L2 flushed (256 MiB fill) before the timed steps and the action "
              "stream (> 126 MiB L2) is read once per row; the recurrent env state (incl. each env's next reset record) and the "
              "output slab stay on chip by construction at this num_envs, re-warmed by the "
              "untimed lead-in steps of the timed chain.  Reference arm: "
              "CPU thread pool, not applicable",
    }



def measured_peak_hbm():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms while the bench runs."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.samples = []
        self.proc = None
        self.t = None
        self.device = device

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.device), f"--query-gpu={self.FIELDS}",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.t = threading.Thread(target=self._pump, daemon=True)
        self.t.start()

    def _pump(self):
        for line in self.proc.stdout:
            self.samples.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons, power = [], None, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.samples:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                smax = float(parts[1])
                if t0 - 0.05 <= ts <= t1 + 0.05:
                    sm.append(float(parts[0]))
                    power.append(float(parts[2]))
                    for nm, v in zip(names, parts[3:7]):
                        if v.lower().startswith("active"):
                            reasons.add(nm)
            except ValueError:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax,
                "reasons": sorted(reasons), "samples_under_load": len(sm),
                "power_w_max": max(power) if power else None}


def bind_to_gpu_numa(local: int):
    """Pin this process (and the pinned host buffers it allocates from now on) to the CPUs of
    the NUMA node the GPU hangs off: a host thread on the far socket pays the inter-socket
    hop on every pinned-memory copy and every doorbell.  Returns what was done."""
    try:
        import torch

        pr = torch.cuda.get_device_properties(local)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as fh:
            node = int(fh.read().strip())
        if node < 0:
            return {"pci": bdf, "node": node, "bound": False}
        with open(f"/sys/devices/system/node/node{node}/cpulist") as fh:
            cpus = set()
            for part in fh.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return {"pci": bdf, "node": node, "bound": False}
        os.sched_setaffinity(0, cpus)
        return {"pci": bdf, "node": node, "bound": True, "cpus": len(cpus)}
    except Exception as exc:  # never fatal: the bench runs unbound
        return {"bound": False, "error": f"{type(exc).__name__}: {exc}"}


def make_action_stream(torch, task, n, device, min_bytes):
    """[T, N, ...] synthetic actions on the device, larger than L2 so no row is re-read
    while it could still be cached."""
    eng, _, _, nact = TASKS[task]
    row = n * (48 if eng == "HalfCheetah" else 4)
    T = max(64, -(-min_bytes // row))
    T = -(-T // 64) * 64
    g = torch.Generator(device=device)
    g.manual_seed(1)
    if eng == "HalfCheetah":
        a = torch.rand((T, n, 6), generator=g, device=device, dtype=torch.float64) * 2 - 1
    elif nact is None:
        a = (torch.rand((T, n, 1), generator=g, device=device, dtype=torch.float32) * 4 - 2)
    else:
        a = torch.randint(0, nact, (T, n), generator=g, device=device, dtype=torch.int32)
    return a


class Timer:
    """Timed chains of one pool.  A chain of `lead + K` steps is captured once; its two
    timestamps sit INSIDE the graph (epb_step_many_timed): from the moment step `lead` became
    ready to the completion of step `lead + K - 1` -- exactly K steps in the chain's steady
    state, no host launch latency in the window whatever K is.  K above MAX_CHAIN is cut
    into MAX_CHAIN-step chains that are timed one after the other and summed."""

    def __init__(self, torch, dist, pool, actions, dev, world, use_graph=True):
        self.torch, self.dist, self.pool, self.actions = torch, dist, pool, actions
        self.dev, self.world, self.use_graph = dev, world, use_graph
        self.flush = torch.empty(2 * L2_BYTES, dtype=torch.uint8, device=dev)
        self.launches = 0

    def _one(self, K, lead, exchange, warm):
        pool, torch = self.pool, self.torch
        if exchange:   # chain length a multiple of the ring depth: replays reuse one graph
            lead += (-(lead + K)) % max(pool.exchange_depth, 1)
        n_chain = lead + K
        if warm:  # capture + instantiate + first replay outside every timed window
            pool.step_many_timed(self.actions, 0, n_chain, lead, n_chain, exchange,
                                 self.use_graph)
        with torch.cuda.stream(torch.cuda.ExternalStream(pool.stream, device=self.dev)):
            self.flush.fill_(1)
        torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        l0 = pool.launch_count
        ms = pool.step_many_timed(self.actions, 0, n_chain, lead, n_chain, exchange,
                                  self.use_graph)
        self.launches += round((pool.launch_count - l0) * K / n_chain)
        return ms

    def run(self, K, lead, exchange=False):
        """Total milliseconds of K timed steps on this rank, then the MAX over ranks."""
        self.launches = 0
        total, left, first = 0.0, K, True
        while left > 0:
            k = min(left, MAX_CHAIN)
            total += self._one(k, lead, exchange, warm=first or k != MAX_CHAIN)
            left -= k
            first = False
        if self.world > 1:
            tt = self.torch.tensor([total], device=self.dev, dtype=self.torch.float64)
            self.dist.all_reduce(tt, op=self.dist.ReduceOp.MAX)
            total = float(tt.item())
        return total


def attach_exchange(torch, dist, pool, world, rank, dev):
    """Collective: allocate the ring, swap CUDA IPC handles, map the peers.  Returns an
    error string (on every rank) or None."""
    def all_ok(ok):
        f = torch.tensor([1 if ok else 0], device=dev, dtype=torch.int32)
        dist.all_reduce(f, op=dist.ReduceOp.MIN)
        return bool(f.item())

    err, handle = "", None
    try:
        handle = pool.exchange_init(world, rank)
    except Exception as exc:
        err = f"exchange_init: {exc}"
    if not all_ok(handle is not None):
        return err or "a peer failed exchange_init"
    handles = [None] * world
    dist.all_gather_object(handles, handle)
    try:
        pool.exchange_attach_ipc(handles)
    except Exception as exc:
        err = f"exchange_attach_ipc: {exc}"
    if not all_ok(not err):
        return err or "a peer failed exchange_attach_ipc"
    dist.barrier()
    return None


def wire_bytes_per_env(pool):
    """Bytes that cross NVLink per env-step and peer: env keys + reward + one packed word."""
    return sum(k.row_bytes for k in pool.keys[8:]) + 4 + 4


def measure_exchange(torch, dist, timer, pool, world, rank, dev, K, lead):
    """`K` exchanged steps (step -> wire columns into every peer -> flags -> receiver-side
    re-expansion), pushes and waits on parallel graph branches: up to depth-1 steps run ahead of
    the batch that is still arriving.  A step counts as complete when its batch has arrived."""
    err = attach_exchange(torch, dist, pool, world, rank, dev)
    if err:
        return {"unavailable": err}
    pool.step_exchange(None)          # forced reset through the exchange: ring primed
    pool.exchange_wait()
    pool.sync()
    ms = timer.run(K, lead, exchange=True)
    pushed, timed_out = pool.exchange_status()
    bad = torch.tensor([1 if timed_out else 0], device=dev, dtype=torch.int32)
    dist.all_reduce(bad, op=dist.ReduceOp.MAX)
    if bad.item():
        return {"unavailable": "a peer wait hit its time bound"}
    wire = wire_bytes_per_env(pool) * pool.n * (world - 1)
    return {"value": pool.n * world * K / (ms * 1e-3), "unit": "env-steps/s", "steps": K,
            "ms_per_step": ms / K, "gpu_launches": timer.launches,
            "nvlink_bytes_in_per_gpu_per_step": wire,
            "nvlink_gbs_in_per_gpu": wire * K / (ms * 1e-3) / 1e9,
            "wire_bytes_per_env_step": wire_bytes_per_env(pool),
            "ring_depth": pool.exchange_depth,
            "api": "epb_step_exchange_many_device: per step the step kernel (writes its slice into "
                   "its ring slot), one push kernel on one of three push branches (checks the ring "
                   "credit, forwards env keys + reward + packed word to every peer over NVLink, "
                   "publishes the slot's flag) and one wait kernel (acquires every peer's flag, "
                   "re-expands the common columns); CUDA-graph replay; pushes, waits and record "
                   "refills on parallel branches"}


def run_allgather(args, torch, dist, pool, actions, dev, world):
    """Library baseline: every step followed by ONE ncclAllGather of the packed output slab
    (all 13 columns), CUDA-graph replayed in 64-step chunks."""
    from envpool_b200._capi import _torch_view
    from envpool_b200.sharded import all_gather_packed

    n, T = pool.n, actions.shape[0]
    slab = _torch_view(pool.outputs_device_ptr(), (pool.slab_bytes,), torch.uint8, dev.index)
    full = torch.empty((world, pool.slab_bytes), dtype=torch.uint8, device=dev)
    steps = int(min(max(args.steps, 64), 512)) // 64 * 64
    chunk = 64
    side = torch.cuda.Stream(device=dev)

    def body(k0):
        for k in range(chunk):
            pool.step_device(actions[(k0 + k) % T],
                             stream=torch.cuda.current_stream(dev).cuda_stream)
            all_gather_packed(slab, full)

    mode = "cuda-graph replay of 64-step chunks"
    with torch.cuda.stream(side):
        body(0)
        torch.cuda.synchronize()
        graph = None
        try:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                body(0)
            graph = g
        except Exception as exc:  # capture unsupported: fall back to eager launches
            mode = f"eager launches (graph capture failed: {type(exc).__name__})"
            torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if graph is not None:
            graph.replay()      # untimed lead-in, no host sync before the timed replays
        ev0.record(side)
        for c in range(steps // chunk):
            if graph is not None:
                graph.replay()
            else:
                body(c * chunk)
        ev1.record(side)
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    tt = torch.tensor([ms], device=dev, dtype=torch.float64)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms = float(tt.item())
    gathered = pool.slab_bytes * (world - 1)
    return {"value": n * world * steps / (ms * 1e-3), "unit": "env-steps/s", "steps": steps,
            "ms_per_step": ms / steps, "allgather_bytes_in_per_gpu_per_step": gathered,
            "nvlink_gbs_in_per_gpu": gathered * steps / (ms * 1e-3) / 1e9,
            "api": "step_device + one ncclAllGather of the packed output slab per step; " + mode}


def roofline_of(pool, eng, n, ms_per_step, task, precision):
    peak, peak_src = measured_peak_hbm()
    bpe = pool.bytes_per_env_step
    achieved = bpe * n / (ms_per_step * 1e-3) / 1e9
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic = json.load(f).get(f"{task}:{n}:{precision}")
    except Exception:
        pass
    hc = {"thread": "hc_thread_kernel", "warp": "hc_kernel"}.get(
        os.environ.get("ENVPOOL_B200_HC_KERNEL", ""), "hc_pair_kernel")
    kern = hc if eng == "HalfCheetah" else "step_kernel<%s>" % eng
    out = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
           "frac": achieved / peak, "traffic": traffic, "bytes_per_env_step": bpe,
           "peak_source": peak_src, "kernel": kern}
    if eng == "HalfCheetah":
        out["note"] = ("compute-bound (SURVEY 8d): the HBM fraction is reported as required; "
                       "see `compute`")
        try:
            from envpool_b200 import _capi

            with open(os.path.join(ROOT, "profiles", "hc_flops.json")) as f:
                hc = json.load(f)
            flop = float(hc["fp64_flop_per_env_step"])
            pk = _capi.fp64_peak_gflops(pool.device)
            ach = flop * n / (ms_per_step * 1e-3) / 1e9
            out["compute"] = {"bound": "fp64", "achieved": ach, "peak": pk, "unit": "GFLOP/s",
                              "frac": ach / pk, "flop_per_env_step": flop,
                              "peak_source": "measured live: epb_fp64_peak_gflops (8 independent "
                                             "DFMA chains per thread)",
                              "flop_source": hc.get("source", "profiles/hc_flops.json")}
        except Exception as exc:
            out["compute"] = {"error": f"{type(exc).__name__}: {exc}"}
    return out


def run_config_line(torch, dist, task, n_total, world, rank, local, dev, steps, lead, label):
    """One BASELINE.json config at this --gpus: n_total envs sharded over the ranks (strong
    scaling: the total is what the config names).  Step-only and, at N>1, with the exchange."""
    from envpool_b200 import _capi

    eng, ms_, iopt, _ = TASKS[task]
    n = n_total // world
    pool = _capi.CPool(eng, n, seed=0, max_episode_steps=ms_, iopt=iopt, device=local,
                       env_id_offset=rank * n)
    actions = make_action_stream(torch, task, n, dev, 2 * L2_BYTES)
    timer = Timer(torch, dist, pool, actions, dev, world)
    pool.reset_device()
    pool.step_many_device(actions, 0, min(16, steps))
    pool.sync()
    ms = timer.run(steps, lead)
    line = {"config": label, "task": task, "num_envs_total": n_total, "num_envs_per_gpu": n,
            "n_gpus": world, "steps": steps, "unit": "env-steps/s",
            "replicas": {"value": n_total * steps / (ms * 1e-3), "ms_per_step": ms / steps},
            "roofline": roofline_of(pool, eng, n, ms / steps, task, "f64")}
    line["value"] = line["replicas"]["value"]
    line["value_is"] = "step only (1 GPU: nothing to exchange)"
    if world > 1:
        px = measure_exchange(torch, dist, timer, pool, world, rank, dev, steps, lead)
        line["with_exchange"] = px
        if "value" in px:
            line["value"] = px["value"]
            line["value_is"] = "with the engine's peer exchange"
    pool.close()
    del actions, timer
    torch.cuda.empty_cache()
    return line


def dump_outputs(pool, path):
    """The output columns of `pool`'s last step, as a caller of the device path receives them,
    to path/<key>.npy: float columns as they are, integer columns as float64, flags as
    float32.  Above DUMP_BYTES only a fixed, seeded sample of env rows is written (the same
    rows in every run; the info:env_id column says which)."""
    cols = {k: v.cpu().numpy() for k, v in pool.outputs_torch().items()}
    cols = {k: v if v.dtype.kind == "f" else v.astype(np.float64 if v.dtype.kind in "iu"
                                                       else np.float32)
            for k, v in cols.items()}
    row = sum(v[0].nbytes for v in cols.values())
    if row * pool.n > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(pool.n, DUMP_BYTES // row,
                                                       replace=False))
        cols = {k: v[keep] for k, v in cols.items()}
    os.makedirs(path, exist_ok=True)
    for k, v in cols.items():
        np.save(os.path.join(path, k + ".npy"), v)


def run_ours(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the env-step engine has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa(local) if args.bind else {"bound": False}
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from envpool_b200 import _capi

    eng, ms, iopt, _ = TASKS[args.task]
    n = args.num_envs
    pool = _capi.CPool(eng, n, seed=0, max_episode_steps=ms, iopt=iopt, device=local,
                       precision=args.precision, env_id_offset=rank * n)
    actions = make_action_stream(torch, args.task, n, dev, 2 * L2_BYTES)
    K, W = args.steps, args.warmup
    use_graph = not args.no_graph
    # untimed steps in front of the timed ones, same graph.  128 = several episode lengths of a
    # random-policy CartPole: after the L2 flush every env has reset at least once, i.e. the
    # recurrent on-chip state (env state AND the head of each env's reset-record ring) is back
    # where a long-running loop keeps it before the clock starts.
    lead = int(min(max(W, 128), 256))
    timer = Timer(torch, dist, pool, actions, dev, world, use_graph)

    pool.reset_device()
    pool.sync()
    sampler = ClockSampler(local)
    if rank == 0 and not args.profile:
        sampler.start()
    t_load0 = time.time()
    pool.step_many_device(actions, 0, W, use_graph=False)   # W warm-up steps, direct launches
    pool.sync()
    if not args.profile:
        # ~1 s of the same launches before the timed region: clocks are sampled under load.
        # The env state is put back afterwards, so that what the timed steps compute does not
        # depend on how many steps fit into that second.
        snapshot = pool.state_export()
        t_w = time.time()
        while time.time() - t_w < 1.0:
            pool.step_many_device(actions, 0, min(1024, actions.shape[0]), use_graph=use_graph)
            pool.sync()
        pool.state_import(snapshot)
        del snapshot
    ms_total = timer.run(K, lead)
    launches = timer.launches
    if args.dump_outputs and rank == 0:
        dump_outputs(pool, args.dump_outputs)
    t_load1 = time.time()
    clocks = sampler.stop(t_load0, t_load1) if rank == 0 and not args.profile else None
    ms_per_step = ms_total / K
    replicas = {"value": n * world * K / (ms_total * 1e-3), "ms_per_step": ms_per_step,
                "gpu_launches": int(launches),
                "api": "device-resident C-ABI single-step kernel, one launch per step (+ one "
                       "refill launch beside the next step), no data-path collective"}
    px = ag = None
    if world > 1 and not args.profile:
        ag = run_allgather(args, torch, dist, pool, actions, dev, world)
        px = measure_exchange(torch, dist, timer, pool, world, rank, dev, K, lead)
    result = None
    if rank == 0:
        result = {
            "metric": METRIC, "value": replicas["value"], "unit": "env-steps/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64" if args.precision == "f64" else "f32", "data": "synthetic",
            "config": bench_config(args.task, n, world, args.precision),
            "api": replicas["api"] + (", CUDA-graph replay" if use_graph else ""),
            "timing": f"two timestamps inside one captured chain of {lead} untimed + "
                      f"{min(K, MAX_CHAIN)} timed steps (epb_step_many_timed): from step "
                      f"{lead} becoming ready to the completion of the last step; W={W} "
                      f"direct warm-up launches and ~1 s of replays before; MAX over ranks",
            "value_is": "step only (1 GPU: nothing to exchange)",
            "gpu_launches": int(launches),
            "roofline": roofline_of(pool, eng, n, ms_per_step, args.task, args.precision),
            "clocks": clocks,
            "host": {"numa": numa, "cpus": os.cpu_count()},
        }
        if world > 1:
            result["replicas"] = replicas
            result["with_allgather_nccl"] = ag
            result["with_exchange"] = px
            if px and "value" in px:
                # north_star's path at N > 1 includes the exchange: that is the headline
                result["value"] = px["value"]
                result["ms_per_step"] = px["ms_per_step"]
                result["gpu_launches"] = int(px["gpu_launches"])
                result["value_is"] = ("with the engine's NVLink peer exchange after every step "
                                      "(every GPU holds all envs' outputs); collective-free "
                                      "figure under `replicas`")
                result["api"] = px["api"]
            else:
                result["value_is"] = ("replicas (no collective): the peer exchange was "
                                      "unavailable -- see with_exchange")
    # ---- fused rollout API: T steps per launch, state in registers ----------------------
    if world == 1 and (not args.profile or args.profile_rollout):
        ro = run_rollout(args, torch, pool, actions, dev)
        if rank == 0:
            result["rollout"] = ro
    # ---- e2e through the public API with host buffers --------------------------------
    if not args.profile:
        e2e = run_e2e(args, torch, local, rank, world)
        if rank == 0:
            result["e2e"] = e2e
    pool.close()
    del actions, timer
    torch.cuda.empty_cache()
    # ---- the other BASELINE.json configs at this --gpus ---------------------------------
    if not args.profile and not args.no_configs:
        lines = []
        for label, task, n_total, steps in (
                ("configs[2] classic_control 1M", "Pendulum-v1", 1 << 20, 200),
                ("configs[2] classic_control 1M", "Acrobot-v1", 1 << 20, 100),
                ("configs[3] toy_text 4M", "FrozenLake-v1", 1 << 22, 100),
                ("configs[3] toy_text 4M", "Catch-v0", 1 << 22, 50),
                ("configs[4] HalfCheetah 32768", "HalfCheetah-v4", 32768, 10)):
            try:
                lines.append(run_config_line(torch, dist, task, n_total, world, rank, local,
                                             dev, steps, 8 if task.startswith("Half") else 32,
                                             label))
            except Exception as exc:   # a config line never takes the headline down
                lines.append({"config": label, "task": task,
                              "error": f"{type(exc).__name__}: {exc}"})
        if rank == 0:
            result["configs"] = lines
    if rank == 0 and world == 1 and not args.profile and not args.no_cpu:
        result["cpu_baseline"] = reference_at_best_threads(args, args.num_envs, steps=None,
                                                           warmup=3, budget_s=args.cpu_seconds)
    if rank == 0:
        print(json.dumps(result))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_rollout(args, torch, pool, actions, dev):
    """epb_rollout_device: T consecutive sync steps of all envs in ONE launch (the fused
    random-action rollout of north_star); every step's outputs are written to [T, N, ...]
    arrays in HBM, actions are read from the [T, N] stream, env state lives in registers."""
    n = pool.n
    out_row = sum(k.row_bytes for k in pool.keys)
    T = int(max(4, min(64, (2 << 30) // max(1, out_row * n), actions.shape[0])))
    tdt = {np.dtype(np.int32): torch.int32, np.dtype(np.float32): torch.float32,
           np.dtype(np.float64): torch.float64, np.dtype(np.bool_): torch.bool}
    cols = [torch.empty((T, n) + k.shape, dtype=tdt[k.dtype], device=dev) for k in pool.keys]
    stream = torch.cuda.ExternalStream(pool.stream, device=dev)
    launches = max(3, min(200, args.steps // T))
    nrows = actions.shape[0] // T
    for i in range(3):
        pool.rollout_device(actions[(i % nrows) * T:], T, cols)
    pool.sync()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for i in range(launches):
        pool.rollout_device(actions[(i % nrows) * T:], T, cols)
    ev1.record(stream)
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    steps = launches * T
    state_bytes = pool.bytes_per_env_step - pool.action_key.row_bytes - out_row
    bpe = pool.action_key.row_bytes + out_row + state_bytes / T
    peak, _ = measured_peak_hbm()
    achieved = bpe * n * steps / (ms * 1e-3) / 1e9
    return {"value": n * steps / (ms * 1e-3), "unit": "env-steps/s", "T_per_launch": T,
            "launches": launches, "ms_per_step": ms / steps,
            "bytes_per_env_step": bpe,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak},
            "api": "epb_rollout_device: T steps per launch, outputs [T,N,...] written to HBM"}


def run_e2e(args, torch, local, rank, world):
    """Same metric through envpool_b200.make(...).step(numpy): per step the action batch is
    copied host->device (via pinned staging) and every state column comes back device->host
    into a pinned slab that the returned numpy arrays view."""
    import envpool_b200

    eng, ms, iopt, nact = TASKS[args.task]
    n = args.num_envs
    env = envpool_b200.make(args.task, env_type="gymnasium", num_envs=n, seed=0,
                            device=local, precision=args.precision, env_id_offset=rank * n)
    rng = np.random.default_rng(1)
    Ta = 64
    if eng == "HalfCheetah":
        acts = rng.uniform(-1, 1, size=(Ta, n, 6))
    elif nact is None:
        acts = rng.uniform(-2, 2, size=(Ta, n, 1)).astype(np.float32)
    else:
        acts = rng.integers(0, nact, size=(Ta, n)).astype(np.int32)
    env.reset()
    E = int(min(max(args.steps, 50), 400))
    for t in range(20):   # warm-up holds its results exactly like the timed loop
        obs, rew, term, trunc, info = env.step(acts[t % Ta])
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    checksum = 0.0
    for t in range(E):
        obs, rew, term, trunc, info = env.step(acts[t % Ta])
        checksum += float(rew[0])
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if world > 1:
        import torch.distributed as dist
        tt = torch.tensor([dt], device=f"cuda:{local}", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
    dp = env.device_pool
    # the two id columns of a full identity batch are constants already held by the pinned
    # slab: the D2H copy starts at the third column
    d2h = int(dp.slab_bytes - dp.keys[2].offset)
    return {"value": n * world * E / dt, "unit": "env-steps/s", "steps": E,
            "h2d_bytes_per_step": int(acts[0].nbytes) * world,
            "d2h_bytes_per_step": d2h * world,
            "ms_per_step": dt / E * 1e3,
            "api": "envpool_b200.make(task,'gymnasium').step(numpy actions) -> numpy"}


def _ref_actions(eng, nact, n, rng, Ta=16):
    if eng == "HalfCheetah":
        return rng.uniform(-1, 1, size=(Ta, n, 6))
    if nact is None:
        return rng.uniform(-2, 2, size=(Ta, n, 1)).astype(np.float32)
    return rng.integers(0, nact, size=(Ta, n)).astype(np.int32)


def cpu_baseline(args, n, budget_s=15.0, steps=None, warmup=3, num_threads=0):
    """The reference's own CPU thread pool (oracle/_ref = its AsyncEnvPool + env headers
    compiled from /root/reference) stepping an n-env batch on this box's host cores; falls
    back to the scalar oracle port when _ref is absent (HalfCheetah: no MuJoCo here)."""
    eng, ms, iopt, nact = TASKS[args.task]
    rng = np.random.default_rng(1)
    from oracle import ref_lib

    cores = os.cpu_count() or 1
    if ref_lib.available() and eng != "HalfCheetah":
        acts = _ref_actions(eng, nact, n, rng)
        pool = ref_lib.RefPool(eng, n, seed=0, max_episode_steps=ms, iopt=iopt,
                               num_threads=num_threads)
        if steps is None:
            probe = pool.bench(acts, 1, 3) / 3
            steps = int(min(max(budget_s / max(probe, 1e-6), 10), 5000))
        dt = pool.bench(acts, warmup, steps)
        pool.close()
        used = min(n, cores) if num_threads <= 0 else num_threads
        return {"value": n * steps / dt, "unit": "env-steps/s", "cores": used,
                "kind": "reference", "ms_per_step": dt / steps * 1e3,
                "sample": f"{steps} sync steps of a {n}-env batch, AsyncEnvPool "
                          f"num_threads={used} of {cores} hw threads"
                          + (" (its default: min(batch, hw threads))" if num_threads <= 0
                             else "")}
    from oracle.oracle_lib import OraclePool

    pool = OraclePool(eng, n, seed=0, max_episode_steps=ms, iopt=iopt)
    acts = _ref_actions(eng, nact, n, rng, 4)
    pool.reset()
    t0 = time.perf_counter()
    pool.step(acts[0])
    probe = time.perf_counter() - t0
    if steps is None:
        steps = int(min(max(budget_s / max(probe, 1e-6), 2), 2000))
    t0 = time.perf_counter()
    for t in range(steps):
        pool.step(acts[t % 4])
    dt = time.perf_counter() - t0
    return {"value": n * steps / dt, "unit": "env-steps/s", "cores": 1, "kind": "port",
            "ms_per_step": dt / steps * 1e3,
            "sample": f"{steps} sync steps of a {n}-env batch, scalar C port"}


def sweep_reference_threads(args, n, steps=10):
    """The reference's default thread count (every hardware thread) is not its best on a
    many-core host: each dequeue is serialised by one semaphore
    (action_buffer_queue.h:71-80) and the workers spin.  Its own benchmark script takes
    num_threads as a knob (benchmark/test_envpool.py), so give it the best of a sweep -- on
    the REAL batch (n envs), `steps` (>= 10) steps per count; a count whose 2-step probe is
    already 3x slower than the best so far is not run to the end.
    Returns (best num_threads (0 = the default), {threads: env-steps/s})."""
    from oracle import ref_lib

    eng = TASKS[args.task][0]
    if not ref_lib.available() or eng == "HalfCheetah":
        return 0, {}
    cores = os.cpu_count() or 1
    cand = sorted({max(1, cores // d) for d in (1, 2, 4, 8, 16)} | {8, 16, 24, 32}, reverse=True)
    cand = [c for c in cand if c <= cores]
    cand.sort(key=lambda c: abs(c - 16))   # the usual optimum first: it sets the bar
    sweep, best, best_v = {}, 0, 0.0
    for nt in cand:
        probe = cpu_baseline(args, n, steps=2, warmup=1, num_threads=nt)
        if best_v and probe["value"] * 3 < best_v:
            sweep[str(nt)] = round(probe["value"])
            continue
        r = cpu_baseline(args, n, steps=steps, warmup=1, num_threads=nt)
        sweep[str(nt)] = round(r["value"])
        if r["value"] > best_v:
            best, best_v = nt, r["value"]
    return best, sweep


def reference_at_best_threads(args, n, steps, warmup, budget_s):
    """cpu_baseline at the best thread count of the sweep (never fatal: falls back to the
    reference's default count)."""
    try:
        nt, sweep = sweep_reference_threads(args, n)
    except Exception as exc:
        nt, sweep = 0, {"error": f"{type(exc).__name__}: {exc}"}
    cb = cpu_baseline(args, n, budget_s=budget_s, steps=steps, warmup=warmup, num_threads=nt)
    cb["threads_swept"] = sweep
    return cb


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path (oracle/_ref = its
    AsyncEnvPool + env headers compiled from /root/reference) on this box's host cores, same
    metric / config as our arm.  A "step" is one Send/Recv of a batch; when K full-size
    batches would not finish in a few minutes, each step is a bounded sample of the workload
    (a smaller batch of the same env, same thread count) -- said in `cpu_baseline.sample`."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    K, W = args.steps, args.warmup
    n_full = args.num_envs * world   # our arm at this --gpus steps this many envs per step
    budget_s = 120.0
    # per-env-step cost at a moderate thread count, to size the per-step sample
    probe = cpu_baseline(args, min(n_full, 65536), steps=3, warmup=1, num_threads=16)
    rate = max(probe["value"], 1.0)
    n_s = int(min(n_full, max(64, rate * budget_s / max(K + W, 1))))
    if n_s < n_full:
        n_s = 1 << (n_s.bit_length() - 1)   # power of two, >= 64
    cb = reference_at_best_threads(args, n_s, steps=K, warmup=W, budget_s=budget_s)
    if n_s < n_full:
        cb["sample"] = (f"each of the {K} steps is a {n_s}-env batch (bounded sample of the "
                        f"{n_full}-env workload so that the run ends in minutes); "
                        + cb["sample"])
    out = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "env-steps/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": cb["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": bench_config(args.task, args.num_envs, world, args.precision),
        "api": f"the reference's AsyncEnvPool (C++ Send/Recv loop, benchmark/test_envpool.py "
               f"pattern) on {cb['cores']} host threads",
        "note": "the reference has no GPU path; one process uses the host cores, so the value "
                "does not scale with --gpus",
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default: 20000; 100 with --impl reference)")
    ap.add_argument("--warmup", type=int, default=None,
                    help="untimed warm-up steps (default: 2000; 3 with --impl reference)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--task", default="CartPole-v1", choices=sorted(TASKS))
    ap.add_argument("--num-envs", type=int, default=65536, help="envs per GPU")
    ap.add_argument("--precision", default="f64", choices=["f64", "f32"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-configs", action="store_true",
                    help="skip the lines for BASELINE.json configs 3-5")
    ap.add_argument("--bind", action="store_true",
                    help="bind the process to the GPU's NUMA node (measured: no gain on the "
                         "pool's 2-socket hosts, profiles/r2_e2e.md)")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--profile", action="store_true",
                    help="kernel loop only (for ncu): no clocks sampler, e2e or cpu legs")
    ap.add_argument("--profile-rollout", action="store_true",
                    help="with --profile: also run the fused rollout leg (for ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<key>.npy")
    args = ap.parse_args()
    ref = args.impl == "reference"
    if args.steps is None:
        args.steps = 100 if ref else 20000
    if args.warmup is None:
        args.warmup = 3 if ref else 2000
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if ref and args.dump_outputs:
        ap.error("--dump-outputs records our arm's outputs: not with --impl reference")
    if ref:
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
