#!/usr/bin/env python
"""bench.py -- headline benchmark of the batch SGP4/SDP4 path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload config2|config3|config4]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path over the synthetic grid (BASELINE config 2 by default: 13,478
near-earth satellites x 1,440 epochs, fp64, velocities on, TEME).  One JSON line is printed by rank 0.

  value        whole-job props/s with the result left in HBM (CUDA events on the launching stream, max over
               ranks).  N = 1: the whole grid on one GPU.  N > 1 (torchrun, one rank per GPU): the SAME catalog,
               satellite-sharded over the ranks (strong scaling, tile-aligned equal shards, no data-path
               collective) -- "the 13,478 x 1,440 grid at 1, 2, 4 and 8 GPUs" of the north star.  The north star's
               single all-gather of the position/velocity block is timed separately under "allgather": kernel +
               one ncclAllGather, and the fused kernel that stores every run straight into each GPU's copy of the
               block over NVLink; the two gathered blocks are compared bit for bit over every element.
  e2e          the same metric through the reference-facing host-buffer API (Constellation.propagate: host jd/fr
               in, host pos/vel out, copies inside the timed region); "legs" adds the reference's own default
               call shapes (time-major pos+vel = SatrecArray.sgp4; ECEF positions only = astroz.propagate) and
               caller-owned pageable buffers.
  roofline     algorithmic fp64 FLOPs (578 per near-earth cell, SURVEY.md 8a/8d) / kernel time against the fp64
               pipe peak (the larger of the arithmetic peak at the maximum SM clock and a live DFMA
               microbenchmark); HBM figures beside it.
  cpu_baseline the reference's CPU SIMD path (oracle/simd_baseline.c port) timed on this box's host cores.
  config3 / config4   sub-records for the other BASELINE grids (mixed SGP4/SDP4 at N = 1; the week-long grid
               sharded + gathered at N > 1).
  --impl reference  times only that CPU path and prints the same line shape with "impl": "reference".
  --dump-outputs DIR  after the timed steps, writes the position and velocity blocks of the last timed step as
               DIR/pos.npy and DIR/vel.npy (float64, satellite-major TEME, km and km/s): the rows dump_rows() picks, a
               fixed seeded sample when the whole block would not fit DUMP_BYTES.  The workloads are seeded, so two
               builds (or the two --impl arms) can be compared cell for cell.  One process only (--gpus 1).
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
sys.path.insert(0, ROOT)

FLOP_PER_CELL = 578.0          # SURVEY.md section 8a: 387 + 43*K (K=4), div = sqrt = 1
# SURVEY.md section 8a, Sdp4Batch row: ~1.0 kFLOP per non-resonant deep-space cell, ~1.5 kFLOP per resonant one,
# both including the shared Kepler/short-period core at K = 4 (the survey's estimate from op counts)
FLOP_PER_SDP4_CELL = {0: 1000.0, 1: 1500.0, 2: 1500.0}
BYTES_PER_CELL = 48.2          # 48 B written (pos+vel) + ~0.2 B of element reads
PUBLISHED_CPU_HEADLINE = 303e6  # props/s, astroz 16 threads on Ryzen 7 7840U (README.md:39)
METRIC = "propagations/sec (sat x time pairs)"
DUMP_BYTES = 48_000_000        # pos + vel written by --dump-outputs, float64: well under 64 MB


def dump_rows(n_sats: int, n_times: int) -> np.ndarray:
    """Satellite rows --dump-outputs writes: all of them when pos + vel fit DUMP_BYTES, else a sorted sample drawn
    with seed 0 (config2: 694 of the 13,478 rows, every epoch)."""
    k = min(n_sats, max(1, DUMP_BYTES // (2 * n_times * 3 * 8)))
    if k == n_sats:
        return np.arange(n_sats)
    return np.sort(np.random.default_rng(0).choice(n_sats, k, replace=False))


def write_outputs(out_dir: str, pos: np.ndarray, vel: np.ndarray) -> None:
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("pos", pos), ("vel", vel)):
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i",
                 str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                pw.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": max(pw) if pw else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def workload(name: str):
    """(tles, jd, fr, description) of a BASELINE grid.  Every rank of a multi-GPU run builds the SAME catalog."""
    from astroz_b200 import synth

    if name == "config2":
        tles = synth.near_earth_catalog(synth.HEADLINE_SATS, seed=13478)
        jd, fr = synth.time_grid(1440)
        desc = "config2: 13,478 near-earth sats x 1,440 epochs (1-min steps), SGP4, fp64, velocities on, TEME"
    elif name == "config3":
        tles = synth.mixed_catalog(synth.HEADLINE_SATS, seed=28626)
        jd, fr = synth.time_grid(1440)
        desc = "config3: 13,478 sats (1,024 GEO + 256 Molniya + 256 GPS-like deep-space) x 1,440 epochs, mixed SGP4/SDP4"
    elif name == "config4":
        tles = synth.near_earth_catalog(synth.HEADLINE_SATS, seed=13478)
        jd, fr = synth.time_grid(10080)
        desc = "config4: 13,478 near-earth sats x 10,080 epochs (1 week @ 1 min)"
    else:
        raise SystemExit(f"unknown workload {name}")
    return tles, jd, fr, desc


# ------------------------------------------------------------------------------------------------------
def usable_cpus() -> dict:
    """Threads the CPU arm can really run at once: logical CPUs, narrowed by the affinity mask and by the cgroup CPU
    quota of the container (the pool's boxes show 128 logical CPUs under a 16-CPU quota: 128 threads there are
    throttled to a third of the rate 16 threads sustain)."""
    info = {"logical": os.cpu_count() or 1, "affinity": len(os.sched_getaffinity(0)), "cgroup_cpu_max": None}
    n = min(info["logical"], info["affinity"])
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        info["cgroup_cpu_max"] = f"{quota} {period}"
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period) + 0.5)))
    except (OSError, ValueError):
        pass
    info["threads"] = n
    return info


def cpu_reference_pass(tles, jd, fr, min_seconds: float, min_reps: int, max_reps: int, sdp4_threads: int = 0):
    """Time the CPU SIMD port (restatement of src/Sgp4Batch.zig + src/Sdp4Batch.zig + src/Constellation.zig threading)
    on all host threads, outputs pre-touched so page faults are not billed to either arm.  Also returns the time-major
    (pos, vel) block of the last pass."""
    from oracle import oracle as orc

    orc.build()
    sim = orc.SimdConstellation(tles)
    n, nt = len(tles), len(jd)
    pos = np.zeros((nt, n, 3))
    vel = np.zeros((nt, n, 3))
    threads = int(os.environ.get("ASTROZ_THREADS", usable_cpus()["threads"]))   # src/Constellation.zig:61-74
    sim.propagate(jd[:32], fr[:32], layout=1, threads=threads, out=(pos[:32], vel[:32]), sdp4_threads=sdp4_threads)
    times = []
    t_end = time.perf_counter() + min_seconds
    while len(times) < min_reps or (time.perf_counter() < t_end and len(times) < max_reps):
        t0 = time.perf_counter()
        sim.propagate(jd, fr, layout=1, threads=threads, out=(pos, vel), sdp4_threads=sdp4_threads)
        times.append(time.perf_counter() - t0)
    return times, threads, orc.simd_isa(), sim.numSdp4, (pos, vel)


def cpu_baseline_record(tles, jd, fr, seconds: float, min_reps: int, max_reps: int) -> dict:
    """cpu_baseline for one workload.  A catalog with deep-space members is timed under both thread policies of
    the SDP4 phase -- the reference's own (the phase gets the threads the SGP4 phase left over, i.e. one,
    src/Constellation.zig:358-364) and an even split -- and the FASTER one is the baseline."""
    cells = len(tles) * len(jd)
    times, threads, isa, nd, _ = cpu_reference_pass(tles, jd, fr, seconds, min_reps, max_reps, 0)
    rec = {"value": cells * len(times) / sum(times), "unit": "props/s", "cores": threads, "kind": "port", "isa": isa,
           "host": usable_cpus(),
           "sample": f"full grid ({cells} cells) x {len(times)} passes over ~{sum(times):.0f} s, sustained mean, "
                     "time-major, velocities on, outputs pre-touched, one thread per usable CPU",
           "best_pass_value": cells / min(times),
           "published_reference": "303 M props/s (16 thr) / 37.7 M (1 thr) on Ryzen 7 7840U, README.md:39 (near-earth only)"}
    if nd:
        t2, _, _, _, _ = cpu_reference_pass(tles, jd, fr, seconds, min_reps, max_reps, max(1, threads // 2))
        even = cells * len(t2) / sum(t2)
        rec["sdp4_thread_policy"] = {"reference_rule_value": rec["value"], "even_split_value": even,
                                     "note": "src/Constellation.zig:358-364 gives the deep-space phase only the threads "
                                             "the near-earth phase left over (one); the faster policy is reported"}
        if even > rec["value"]:
            rec["value"] = even
            rec["best_pass_value"] = cells / min(t2)
    return rec


def run_reference(args, rank: int, world: int) -> None:
    if rank != 0:
        return
    tles, jd, fr, desc = workload(args.workload)
    cells = len(tles) * len(jd)
    reps = args.warmup + args.steps
    times, threads, isa, nd, (pos, vel) = cpu_reference_pass(tles, jd, fr, 0.0, reps, reps, 0)
    policy = "reference rule"
    if nd:   # mixed catalog: also the even split of threads for the deep-space phase; keep the faster
        t2, _, _, _, _ = cpu_reference_pass(tles, jd, fr, 0.0, reps, reps, max(1, threads // 2))
        if sum(t2[args.warmup:]) < sum(times[args.warmup:]):
            times, policy = t2, "even split of threads between the SGP4 and SDP4 phases"
    if args.dump_outputs:   # threads split satellites, so both policies give the same numbers; block is (nt, n, 3)
        rows = dump_rows(len(tles), len(jd))
        write_outputs(args.dump_outputs, pos[:, rows].transpose(1, 0, 2), vel[:, rows].transpose(1, 0, 2))
    timed = times[args.warmup:]
    total = float(sum(timed))
    value = cells * len(timed) / total
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "props/s", "n_gpus": args.gpus,
        "steps": len(timed), "warmup": args.warmup, "ms_per_step": 1e3 * total / len(timed), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": value / PUBLISHED_CPU_HEADLINE, "dtype": "f64", "data": "synthetic",
        "config": {"workload": desc, "layout": "each arm's faster layout (CPU: time-major, the reference's fast path; "
                                                "GPU: satellite-major)", "isa": isa, "sdp4_thread_policy": policy},
        "cpu_baseline": {"value": value, "unit": "props/s", "cores": threads, "kind": "port", "host": usable_cpus(),
                         "sample": f"full grid ({cells} cells) x {len(timed)} timed passes, outputs pre-touched",
                         "what": "C port of the reference's 8-lane SIMD batch path, SGP4 and SDP4 "
                                 "(Zig 0.16 is not installable here)"},
        "e2e": {"value": value, "unit": "props/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------------------
class Harness:
    """Device, stream, distributed plumbing shared by every leg."""

    def __init__(self, rank: int, local_rank: int, world: int):
        import torch

        self.torch = torch
        self.rank, self.local_rank, self.world = rank, local_rank, world
        self.dist = None
        if world > 1:
            import torch.distributed as dist

            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
                os.environ["NCCL_DEBUG"] = "WARN"   # keep NCCL's banner off stdout: rank 0 prints ONE JSON line
            torch.cuda.set_device(local_rank)
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            self.dist = dist
        torch.cuda.set_device(local_rank)
        self.dev = torch.device("cuda", local_rank)
        self.stream = torch.cuda.Stream(self.dev)   # kernels, events and the collective all go through this stream
        torch.cuda.set_stream(self.stream)

    @classmethod
    def solo(cls, other: "Harness") -> "Harness":
        """The same device and stream, without the collectives: for a leg only one rank runs."""
        me = cls.__new__(cls)
        me.__dict__.update(other.__dict__)
        me.dist = None
        return me

    def barrier(self):
        self.torch.cuda.synchronize(self.dev)
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def rank0_section_done(self, key: str):
        """Rank 0 announces the end of a section it ran alone; the other ranks sleep on the rendezvous store until then.
        (Waiting inside an NCCL barrier instead keeps one host thread per waiting rank spinning in
        cudaStreamSynchronize: seven busy CPUs of the pool's 16-CPU quota while rank 0 drives eight GPUs.)"""
        if self.dist is None:
            return
        import datetime

        store = self.dist.distributed_c10d._get_default_store()
        if self.rank == 0:
            store.set(key, "1")
        else:
            store.wait([key], datetime.timedelta(seconds=1800))

    def max_over_ranks(self, x: float) -> float:
        if self.dist is None:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def all_true(self, ok: bool) -> bool:
        if self.dist is None:
            return ok
        t = self.torch.tensor([1.0 if ok else 0.0], device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return bool(t.item() == 1.0)

    def time_steps(self, fn, steps: int) -> float:
        """ms per step of `fn` queued `steps` times on the launching stream, CUDA events, max over ranks."""
        e0 = self.torch.cuda.Event(enable_timing=True)
        e1 = self.torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record(self.stream)
        for _ in range(steps):
            fn()
        e1.record(self.stream)
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1)) / steps


def e2e_leg(h: Harness, c, jd, fr, rows: int, layout: int, mode: int, velocities: bool, pinned: bool, reps: int,
            total_cells: int, what: str, alloc=None) -> dict:
    """One host-to-host call shape through Constellation.propagate: host time axis in, host result block out, the
    result read on the host every step.  `rows` = satellites of this rank's shard."""
    import astroz_b200

    nt = len(jd)
    shape = (rows, nt, 3) if layout == 0 else (nt, rows, 3)
    buffers = "pinned (astroz_cuda_host_alloc)" if pinned else "caller-owned pageable (numpy)"
    if alloc is not None:
        buffers = "pinned, each GPU's rows on its NUMA node (astroz_cuda_constellation_host_block)"
    elif pinned:
        alloc = astroz_b200.pinned_empty
    else:
        alloc = lambda s: np.zeros(s)   # noqa: E731  zeros: pages touched before the clock
    hp = alloc(shape) if rows else None
    hv = alloc(shape) if (rows and velocities) else None

    def call():
        if c is not None:
            c.propagate(jd, fr, hp, hv, mode, layout, velocities=velocities)
            return float(hp.reshape(-1)[0])
        return 0.0

    for _ in range(2):
        call()
    h.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        checksum = call()
    sec = h.max_over_ranks(time.perf_counter() - t0) / reps
    per_cell = 48 if velocities else 24
    return {"value": total_cells / sec, "unit": "props/s", "ms_per_step": sec * 1e3, "what": what,
            "buffers": buffers,
            "h2d_bytes_per_step": 2 * nt * 8, "d2h_bytes_per_step": total_cells * per_cell,
            "d2h_GBs": total_cells * per_cell / sec / 1e9, "checksum": checksum}


def k2_roofline(c, jd, kernel_ms_k2: float, pipe_peak: float) -> dict:
    """Roofline of the deep-space grid kernel with its own algorithmic FLOP count (SURVEY.md section 8a)."""
    classes = np.asarray(c.classes)
    nt = len(jd)
    flops = sum(FLOP_PER_SDP4_CELL[k - 1] * int((classes == k).sum()) for k in (1, 2, 3)) * nt
    cells = int((classes != 0).sum()) * nt
    ach = flops / (kernel_ms_k2 * 1e-3) / 1e12
    return {"bound": "fp64", "kernel": "sdp4_grid_kernel", "achieved": ach, "peak": pipe_peak, "unit": "TFLOP/s",
            "frac": ach / pipe_peak if pipe_peak else None, "kernel_ms": kernel_ms_k2, "cells": cells,
            "flop_per_cell": {"non_resonant": 1000.0, "resonant": 1500.0, "mean": flops / max(cells, 1)},
            "note": "timed alone (astroz_cuda_sdp4_propagate_into_device); in a mixed call it overlaps the near-earth grid"}


def run_ours(args, rank: int, local_rank: int, world: int) -> None:
    import torch

    import astroz_b200
    from astroz_b200 import Constellation, Layout, OutputMode
    from astroz_b200.parallel import ShardedPropagator, bind_to_gpu_numa_node, shard_rows

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: astroz_b200 has no CPU propagation path")
    # Rank 0's stdout carries exactly ONE JSON line.  NCCL (version banner at communicator creation) and other native
    # libraries write to file descriptor 1 directly, so for the whole run fd 1 points at stderr and the line is written to
    # the saved descriptor at the end.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    h = Harness(rank, local_rank, world)
    dev, stream, dist = h.dev, h.stream, h.dist
    affinity0 = os.sched_getaffinity(0) if world > 1 else None
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None   # host staging next to this GPU's PCIe root

    tles, jd, fr, desc = workload(args.workload)
    n, nt = len(tles), len(jd)
    cells = n * nt                                      # the WHOLE job's cells, whatever N is
    sp = ShardedPropagator(tles, rank, world, device=local_rank, dist=dist)   # tile-aligned equal shards of ONE catalog
    c = sp.local                                        # this rank's constellation (None if its range is empty)
    rows = sp.rows                                      # rows per rank (last rank may hold fewer real satellites)
    n_local = sp.n_local
    n_sdp4_local = c.numSdp4 if c is not None else 0
    kernels_per_step = ((1 if (c is not None and c.numSgp4) else 0) + (1 if n_sdp4_local else 0))

    # NCCL-gather layout: full[r] is rank r's [pos|vel] block, so one in-place ncclAllGather moves everything
    full = torch.empty((world, 2, rows, nt, 3), dtype=torch.float64, device=dev)
    pos, vel = full[rank, 0], full[rank, 1]

    def step():
        if c is not None:
            c.propagate_device(jd, fr, pos, vel, None, OutputMode.teme, Layout.satelliteMajor, out_num_sats=rows,
                               stream=stream.cuda_stream)

    for _ in range(args.warmup):
        step()
    h.barrier()

    # ---- soak: >= 1 s of the same step so the clock sampler sees the device under load, then the timed region ----
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    soak_t0 = time.perf_counter()
    soak_steps = 0
    while time.perf_counter() - soak_t0 < 1.0:
        for _ in range(50):
            step()
        torch.cuda.synchronize(dev)
        soak_steps += 50
    # ---- timed region: exactly K steps, CUDA events on the launching stream, max over ranks ----------------------
    ms_per_step = h.time_steps(step, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:   # the block of the last timed step, before any later leg writes it again
        rows_d = torch.as_tensor(dump_rows(n, nt), device=dev)
        write_outputs(args.dump_outputs, pos.index_select(0, rows_d).cpu().numpy(),
                      vel.index_select(0, rows_d).cpu().numpy())
    if clocks is not None:
        clocks["soak_steps_before_timed_region"] = soak_steps
    value = cells / (ms_per_step * 1e-3)

    # ---- dominant kernel alone (library's own CUDA events around the launch, same stream) ------------------------
    kms, k2ms = [], []
    if c is not None:
        c.set_timing(True)    # CUDA events around the kernels: off in the timed region above (they cost stream time)
    for _ in range(10):
        step()
        torch.cuda.synchronize(dev)
        if c is not None:
            c.synchronize()
            k = c.last_kernel_ms()
            # near-earth only: the events bracketing the one kernel; mixed: the span of the call (its two grids overlap)
            kms.append(k[0] if n_sdp4_local == 0 else (k[1] if k[1] > 0 else k[0] + k[2]))
    kernel_ms_bracketed = h.max_over_ranks(float(np.mean(kms)) if kms else 0.0)
    if c is not None:
        c.set_timing(False)
    # One kernel per step (near-earth catalog): its average launch duration over the timed region IS ms_per_step -- K
    # back-to-back launches between two events -- which is the figure the roofline uses; the per-launch bracketing
    # events of the library add their own ~4 us each and are reported beside it.  A mixed catalog has two overlapping
    # kernels per step: there the bracketed span of the call is the kernel time.
    kernel_ms = ms_per_step if (kernels_per_step == 1 and world == 1) else kernel_ms_bracketed

    # ---- end to end through the host-buffer API -------------------------------------------------------------------
    e2e_steps = max(3, min(args.steps, 10))
    what = ("Constellation.propagate(jd, fr, pos, vel), satellite-major TEME" +
            (f"; one catalog sharded over {world} ranks, every rank copies its rows to its own host block" if world > 1 else ""))
    e2e = e2e_leg(h, c, jd, fr, n_local, 0, 0, True, True, e2e_steps, cells, what)
    legs = {"pinned": e2e}
    legs["pageable"] = e2e_leg(h, c, jd, fr, n_local, 0, 0, True, False, e2e_steps, cells,
                               "same call, caller-owned numpy buffers (what a reference caller passes, "
                               "bindings/python/src/satrec.zig:917-942)")
    legs["time_major_pos_vel"] = e2e_leg(h, c, jd, fr, n_local, 1, 0, True, True, e2e_steps, cells,
                                         "SatrecArray.sgp4 default: time-major (n_times, n_sats, 3) pos+vel "
                                         "(bindings/python/src/satrec.zig:971-982)")
    legs["ecef_positions_only"] = e2e_leg(h, c, jd, fr, n_local, 1, 1, False, True, e2e_steps, cells,
                                          "astroz.propagate() default: ECEF, velocities=False, time-major "
                                          "(bindings/python/astroz/__init__.py:411-413)")

    # ---- N > 1: the same job through ONE handle in ONE process (device = -1: the library fans the call out over the
    # GPUs, each copying its rows over its own PCIe link into one host block).  Rank 0 runs it, the other ranks wait.
    if world > 1:
        h.barrier()
        if rank == 0:
            try:
                if affinity0 is not None:
                    os.sched_setaffinity(0, affinity0)      # the single process serves every GPU: no NUMA pinning
                os.environ["ASTROZ_DEVICES"] = str(world)
                multi = Constellation(tles, device=-1)
                ids, first_rows = multi.devices
                leg = e2e_leg(Harness.solo(h), multi, jd, fr, n, 0, 0, True, True, e2e_steps, cells,
                              f"ONE Constellation handle over {len(ids)} GPUs (device = -1), one process, one propagate call",
                              alloc=lambda shape: multi.host_block(shape[1], 0))
                leg["devices"] = ids
                legs["single_handle_all_gpus"] = leg
                legs["single_handle_all_gpus_plain_pinned"] = e2e_leg(
                    Harness.solo(h), multi, jd, fr, n, 0, 0, True, True, e2e_steps, cells,
                    "same, result blocks from astroz_cuda_host_alloc (all on one NUMA node)")
                del multi
            except Exception as exc:
                legs["single_handle_all_gpus"] = {"unavailable": repr(exc)[:300]}
        h.rank0_section_done("single_handle_leg")
        h.barrier()

    # ---- a device-resident consumer: fused propagate + single-target screen through the host API (N = 1) ----------
    screen = None
    if world == 1 and c.numSdp4 == 0:
        times_min = ((jd + fr) - (jd[0] + fr[0])) * 1440.0
        offs = ((jd[0] + fr[0]) - c.epochs) * 1440.0
        for _ in range(2):
            c.screen_conjunction(times_min, 0, 10.0, epoch_offsets=offs, reference_jd=float(jd[0] + fr[0]))
        h.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            c.screen_conjunction(times_min, 0, 10.0, epoch_offsets=offs, reference_jd=float(jd[0] + fr[0]))
        scr_s = (time.perf_counter() - t0) / e2e_steps
        screen = {"value": cells / scr_s, "unit": "props/s", "ms_per_call": scr_s * 1e3,
                  "d2h_bytes_per_call": 12 * n, "api": "Constellation.screen_conjunction (src/Constellation.zig:683-756)",
                  "note": "same cells propagated, minimum range to one target reduced on the device: host-to-host call "
                          "not bound by PCIe"}

    # ---- the north star's collective, measured apart from `value` --------------------------------------------------
    allgather = None
    config4 = None
    if dist is not None:
        allgather = gather_legs(h, sp, jd, fr, full, step, ms_per_step, cells, max(3, min(args.steps, 10)))
        del full
        torch.cuda.empty_cache()
        if args.workload == "config2":
            config4 = config4_record(h, rank, world, local_rank)

    # ---- config 3 sub-record (N = 1): the mixed SGP4/SDP4 grid with its own kernel roofline and CPU baseline -------
    pipe_peak = max(astroz_b200.fp64_peak_tflops(local_rank), astroz_b200.fp64_pipe_peak_tflops(local_rank))
    config3 = None
    if world == 1 and args.workload == "config2" and not args.no_subrecords:
        config3 = config3_record(h, pipe_peak, args)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- roofline ---------------------------------------------------------------------------------------------------
    peaks, peaks_kind = _peaks()
    live_peak = astroz_b200.fp64_peak_tflops(local_rank)
    arith_peak = astroz_b200.fp64_pipe_peak_tflops(local_rank)
    cells_rank0 = n_local * nt
    ach_tflops = FLOP_PER_CELL * cells_rank0 / (kernel_ms * 1e-3) / 1e12 if kernel_ms else None
    ach_gbs = BYTES_PER_CELL * cells_rank0 / (kernel_ms * 1e-3) / 1e9 if kernel_ms else None
    traffic = None
    tfile = os.path.join(ROOT, "profiles", "traffic.json")   # DRAM bytes per launch from the committed ncu capture
    if os.path.exists(tfile) and world == 1:
        try:
            traffic = json.load(open(tfile)).get(args.workload)
            if isinstance(traffic, dict):
                traffic = traffic.get("total")
        except Exception:
            traffic = None
    roofline = {
        "bound": "fp64", "kernel": "sgp4_grid_kernel" + (" (+ sdp4_grid_kernel side by side)" if n_sdp4_local else ""),
        "achieved": ach_tflops, "peak": pipe_peak, "unit": "TFLOP/s",
        "frac": ach_tflops / pipe_peak if (pipe_peak and ach_tflops) else None,
        "peak_source": "max(arithmetic pipe peak = SMs x 64 DFMA lanes x 2 x max SM clock, live DFMA microbenchmark on this device)",
        "peak_arithmetic": arith_peak, "peak_live_microbenchmark": live_peak,
        "flop_per_cell": FLOP_PER_CELL, "kernel_ms": kernel_ms, "kernel_ms_event_bracketed": kernel_ms_bracketed,
        "kernel_ms_source": ("ms_per_step: one kernel per step, K launches back to back between two CUDA events on the "
                             "launching stream" if (kernels_per_step == 1 and world == 1) else
                             "CUDA events bracketing the launch(es) of one call, mean of 10 calls, max over ranks"),
        "cells_per_launch": cells_rank0,
        "hbm": {"bound": "hbm", "achieved": ach_gbs, "peak": peaks.get("hbm_gbs"), "unit": "GB/s",
                "frac": ach_gbs / peaks["hbm_gbs"] if (peaks.get("hbm_gbs") and ach_gbs) else None,
                "peak_source": peaks_kind, "bytes_per_cell": BYTES_PER_CELL},
        "traffic": traffic,
    }
    if n_sdp4_local:
        roofline["note"] = ("mixed catalog: 578 FLOP/cell is the near-earth figure applied to every cell; the deep-space "
                            "kernel's own roofline (1.0 / 1.5 kFLOP per cell) is under config3.roofline_k2 of the default run")

    # ---- CPU baseline: the reference's SIMD path on this box's host cores (N = 1 only) ------------------------------
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_record(tles, jd, fr, 10.0, 3, 400)

    par = ("one GPU, whole grid" if world == 1 else
           f"ONE 13,478-satellite catalog satellite-sharded x{world} ({rows} rows per rank, tile aligned), "
           "no data-path collective in `value`")
    out = {
        "metric": METRIC, "value": value, "unit": "props/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": value / PUBLISHED_CPU_HEADLINE, "dtype": "f64", "data": "synthetic",
        "config": {"workload": desc, "layout": "each arm's faster layout (CPU: time-major, the reference's fast path; "
                                               "GPU: satellite-major)",
                   "cells_total": cells, "cells_per_gpu": cells_rank0, "n_sats_total": n, "rows_per_rank": rows,
                   "output_bytes_per_step_total": 2 * cells * 24,
                   "l2": f"{2 * cells_rank0 * 24 / 1e6:.1f} MB written per step per GPU"
                         + (" >> 126 MB L2 (nothing re-read between steps)" if 2 * cells_rank0 * 24 > 2 * 126e6 else
                            " (comparable to the 126 MB L2: a step's stores may still be draining while the next runs; "
                            "outputs are write-only, nothing is re-read)")
                         + "; the element table is L2-resident by design",
                   "parallelism": par},
        "e2e": {**e2e, "api": e2e["what"], "numa_binding_rank0": numa, "legs": legs},
        "e2e_screen": screen,
        "gpu_launches": kernels_per_step * args.steps,
        "clocks": clocks,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "baseline_published": {"value": PUBLISHED_CPU_HEADLINE, "what": "astroz CPU SIMD, 16 threads, Ryzen 7 7840U"},
    }
    if allgather is not None:
        out["allgather"] = allgather
    if config3 is not None:
        out["config3"] = config3
    if config4 is not None:
        out["config4"] = config4
    sys.stdout.flush()
    os.write(real_stdout, (json.dumps(out) + "\n").encode())
    if dist is not None:
        dist.destroy_process_group()


def gather_legs(h: Harness, sp, jd, fr, full, step, ms_per_step: float, cells: int, reps: int) -> dict:
    """(a) baseline: shard-local kernel, then ONE in-place ncclAllGather of the [pos|vel] blocks;
    (b) product: the same kernel writes every 768-byte run straight into all GPUs' copies of the block over NVLink 5
        (peer stores into a symmetric allocation), so the transfer overlaps the compute.
    The two gathered blocks are compared over EVERY element (torch.equal), not sampled."""
    from astroz_b200.parallel import SymmetricBlock

    torch, dist, dev, stream = h.torch, h.dist, h.dev, h.stream
    world, rank, rows = h.world, h.rank, sp.rows
    nt = len(jd)

    def nccl():
        step()
        dist.all_gather_into_tensor(full, full[rank])

    for _ in range(2):
        nccl()
    ms_ag = h.time_steps(nccl, reps)
    recv_bytes = (world - 1) * full[0].numel() * 8
    out = {"nccl": {"ms_per_step": ms_ag, "value": cells / (ms_ag * 1e-3),
                    "allgather_only_ms": max(ms_ag - ms_per_step, 0.0),
                    "what": "kernel, then one in-place ncclAllGather of the [pos|vel] blocks (torch.distributed, NCCL)"},
           "recv_GB_per_gpu": recv_bytes / 1e9,
           "what": "every GPU ends with the whole (n_sats, n_times, 3) position and velocity blocks of the ONE catalog"}
    try:
        sym = SymmetricBlock(rows * world, nt, dev)
        c = sp.local

        def fused():
            if c is not None:
                c.propagate_gather(jd, fr, peer_pos=sym.peer_pos, peer_vel=sym.peer_vel, out_num_sats=rows * world,
                                   out_sat_offset=rank * rows, stream=stream.cuda_stream)
            sym.barrier()

        for _ in range(2):
            fused()
        ms_f = h.time_steps(fused, reps)
        # whole-block comparison: NCCL's [rank][pos|vel][rows] against the symmetric [pos|vel][rank*rows + row]
        same = True
        for r in range(world):
            real = max(0, min(sp.n_total - r * rows, rows))   # rows of rank r that hold satellites (padding is never written)
            if real:
                same = same and bool(torch.equal(full[r, :, :real], sym.block[:, r * rows:r * rows + real]))
        out["fused"] = {"ms_per_step": ms_f, "value": cells / (ms_f * 1e-3),
                        "recv_GBs_per_gpu": recv_bytes / 1e9 / (ms_f * 1e-3),
                        "identical_to_nccl": h.all_true(same), "compared": "every element of both gathered blocks (torch.equal)",
                        "multicast_available": sym.has_multicast,
                        "what": "one kernel per GPU: propagate + 128-bit stores of each run into every GPU's copy "
                                "of the block (NVLink 5 peer mappings of a symmetric allocation), then a "
                                "symmetric-memory barrier"}
        del sym
    except Exception as exc:  # symmetric memory unavailable on this box: report, do not hide
        out["fused"] = {"unavailable": repr(exc)[:300]}
    return out


def config4_record(h: Harness, rank: int, world: int, local_rank: int) -> dict:
    """BASELINE config 4: 13,478 x 10,080 (one week at one minute) satellite-sharded over the ranks, results
    all-gathered so every GPU holds the 6.52 GB block -- NCCL and fused, compared over every element."""
    from astroz_b200 import Layout, OutputMode
    from astroz_b200.parallel import ShardedPropagator

    torch, dist, dev, stream = h.torch, h.dist, h.dev, h.stream
    tles, jd, fr, desc = workload("config4")
    n, nt = len(tles), len(jd)
    cells = n * nt
    sp = ShardedPropagator(tles, rank, world, device=local_rank, dist=dist)
    rows, c = sp.rows, sp.local
    full = torch.empty((world, 2, rows, nt, 3), dtype=torch.float64, device=dev)

    def step():
        if c is not None:
            c.propagate_device(jd, fr, full[rank, 0], full[rank, 1], None, OutputMode.teme, Layout.satelliteMajor,
                               out_num_sats=rows, stream=stream.cuda_stream)

    for _ in range(3):
        step()
    ms = h.time_steps(step, 5)
    rec = {"workload": desc + f", satellite-sharded x{world}", "cells_total": cells,
           "value": cells / (ms * 1e-3), "unit": "props/s", "ms_per_step": ms,
           "what": "`value`: shards computed, results left in HBM (no collective); `allgather`: plus the single collective"}
    rec["allgather"] = gather_legs(h, sp, jd, fr, full, step, ms, cells, 3)
    del full
    torch.cuda.empty_cache()
    return rec


def config3_record(h: Harness, pipe_peak: float, args) -> dict:
    """BASELINE config 3 on one GPU: mixed SGP4/SDP4 catalog, device-timed value, the deep-space kernel's own
    roofline, the end-to-end call and the CPU SIMD baseline (Sdp4Batch port)."""
    from astroz_b200 import Constellation, Layout, OutputMode

    torch, dev, stream = h.torch, h.dev, h.stream
    tles, jd, fr, desc = workload("config3")
    n, nt = len(tles), len(jd)
    cells = n * nt
    c = Constellation(tles, device=h.local_rank)
    block = torch.empty((2, n, nt, 3), dtype=torch.float64, device=dev)

    def step():
        c.propagate_device(jd, fr, block[0], block[1], None, OutputMode.teme, Layout.satelliteMajor,
                           stream=stream.cuda_stream)

    for _ in range(max(args.warmup, 3)):
        step()
    ms = h.time_steps(step, max(args.steps, 20))
    kms, k1, k2 = [], [], []
    c.set_timing(True)
    for _ in range(10):
        step()
        torch.cuda.synchronize(dev)
        c.synchronize()
        k = c.last_kernel_ms()
        kms.append(k[1]); k1.append(k[0]); k2.append(k[2])
    # the deep-space grid alone (no near-earth grid next to it): its own kernel time for its own roofline
    nd = c.numSdp4
    dblock = torch.empty((2, nd, nt, 3), dtype=torch.float64, device=dev)
    from astroz_b200 import _lib
    import ctypes as C

    alone = []
    for _ in range(8):
        _lib.check(_lib.lib().astroz_cuda_sdp4_propagate_into_device(
            c._h, _lib.dptr(jd), _lib.dptr(fr), nt, C.c_void_p(dblock[0].data_ptr()), C.c_void_p(dblock[1].data_ptr()),
            0, 0, nd, 0, C.c_void_p(stream.cuda_stream)))
        torch.cuda.synchronize(dev)
        c.synchronize()
        alone.append(c.last_kernel_ms()[2])
    k2_alone = float(np.mean(alone[3:]))
    c.set_timing(False)
    rec = {"workload": desc, "cells_total": cells, "n_sgp4": c.numSgp4, "n_sdp4": nd,
           "value": cells / (ms * 1e-3), "unit": "props/s", "ms_per_step": ms,
           "kernel_ms": {"call_span": float(np.mean(kms)), "sgp4_grid_kernel": float(np.mean(k1)),
                         "sdp4_grid_kernel_side_by_side": float(np.mean(k2)), "sdp4_grid_kernel_alone": k2_alone},
           "roofline_k2": k2_roofline(c, jd, k2_alone, pipe_peak),
           "gpu_launches_per_step": 2}
    rec["e2e"] = e2e_leg(h, c, jd, fr, n, 0, 0, True, True, 5, cells,
                         "Constellation.propagate(jd, fr, pos, vel), satellite-major TEME, mixed catalog")
    del block, dblock
    torch.cuda.empty_cache()
    if not args.no_cpu_baseline:
        rec["cpu_baseline"] = cpu_baseline_record(tles, jd, fr, 6.0, 3, 200)
    return rec


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)     # ~0.9 s of device time at 0.45 ms per step
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", default="config2")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-subrecords", action="store_true", help="skip the config3 sub-record of the default N=1 run")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write pos.npy / vel.npy of the last timed step (sampled rows, see dump_rows) to DIR")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes one process's result block: run it with --gpus 1")
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        if world != args.gpus and world == 1 and args.gpus > 1:
            raise SystemExit("launch multi-GPU runs with torch.distributed.run (one rank per GPU)")
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
