#!/usr/bin/env python
"""bench.py — Mpps of the subscriber-dataplane hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload pipeline_imix] [--impl reference] [--dump-outputs DIR]

A *step* is one batch of 2^22 synthetic frames per GPU through the program of
the chosen workload (default: the full pipeline antispoof -> NAT44 -> QoS on
IMIX frames over 10 k subscribers, BASELINE.json configs[3]).  `value` is
whole-job Mpps with frames resident in HBM when the timed region starts
(CUDA events on the library's stream, max over ranks); `e2e` is the same
metric through the C-ABI call with pinned HOST buffers, host<->device copies
inside the timed region.  `--impl reference` times the reference's own eBPF C
(oracle/_ref, or the port where that library is absent) on the host cores.
Prints ONE JSON line.
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

from bng_b200 import workloads as W  # noqa: E402

METRIC = "Mpps"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.05)

    def result(self):
        self.stop_flag = True
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": []}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ---------------------------------------------------------------------------
# CPU arms
# ---------------------------------------------------------------------------
def _oracle_kind():
    from oracle import pyoracle
    if pyoracle.available("reference"):
        return "reference"
    if not pyoracle.available("port"):
        pyoracle.build("port")
    return "port"


def _cpu_worker(args):
    """One host core: its MAC-hash shard of the subscribers, private map set (as the kernel's per-CPU,
    per-RX-queue execution of the eBPF programs), `steps` passes over a bounded sample."""
    workload, n, rank, world, steps, warmup, kind = args
    from oracle.pyoracle import Oracle
    wl = W.BUILDERS[workload](n, rank, world)
    o = Oracle(kind)
    for m, k, v in wl.maps:
        from bng_b200.layouts import as_bytes
        o.update_batch(m, as_bytes(k), as_bytes(v))
    translated = []
    for prog, h, l in wl.prewarm:
        pa = o.arena(h.shape[0] * 64 + 64)
        pa[: h.shape[0] * 64] = h.reshape(-1)
        o.run(prog, pa, l.copy(), wl.now0 - 1, stride=64)
        if wl.derive is not None:
            translated.append(np.array(pa[: h.shape[0] * 64]))
    if wl.derive is not None:
        wl.headers, wl.lens = wl.derive(translated)
    off16, stride, total16 = W.slot16(wl.lens, wl.imix, wl.headers.shape[1])
    arena = o.arena(total16 * 16 + 64)
    hw = wl.headers.shape[1]

    def restore():
        if off16 is None:
            arena[: wl.n * stride].reshape(wl.n, stride)[:, :hw] = wl.headers
        else:
            a16 = arena[: total16 * 16].reshape(total16, 16)
            for g in range(hw // 16):
                a16[off16.astype(np.int64) + g] = wl.headers[:, 16 * g: 16 * g + 16]

    t_total = 0.0
    for s in range(warmup + steps):
        restore()
        lens = wl.lens.copy()
        t0 = time.perf_counter()
        o.run(wl.prog, arena, lens, wl.now0 + s * wl.now_step, off16=off16, stride=stride)
        dt = time.perf_counter() - t0
        if s >= warmup:
            t_total += dt
    return wl.n * steps, t_total


def cpu_run(workload: str, n: int, procs: int, steps: int, warmup: int):
    import multiprocessing as mp
    kind = _oracle_kind()
    jobs = [(workload, n, r, procs, steps, warmup, kind) for r in range(procs)]
    if procs == 1:
        res = [_cpu_worker(jobs[0])]
    else:
        with mp.get_context("fork").Pool(procs) as pool:
            res = pool.map(_cpu_worker, jobs)
    pk = sum(r[0] for r in res)
    tmax = max(r[1] for r in res)
    return pk / tmax / 1e6, kind, tmax


def host_cpus() -> dict:
    """CPUs this process may actually use: the scheduler affinity mask and the cgroup CPU quota, not os.cpu_count()
    (a container on a 128-thread host can be limited to a fraction of it; sizing the reference arm's pool from
    cpu_count() then oversubscribes the quota and makes the CPU arm look slower than the hardware is)."""
    out = {"os_cpu_count": os.cpu_count() or 1}
    try:
        out["sched_affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        out["sched_affinity"] = out["os_cpu_count"]
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = int(txt[0]) / int(txt[1])
            else:
                q = int(txt[0])
                if q > 0:
                    quota = q / int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            break
        except Exception:
            continue
    out["cgroup_quota_cpus"] = None if quota is None else round(quota, 2)
    usable = out["sched_affinity"]
    if quota is not None:
        usable = max(1, min(usable, int(quota)))
    out["usable"] = usable
    return out


PROGRAM_OF = {"pipeline_imix": "pipeline_up", "pipeline_64": "pipeline_up", "antispoof_64": "antispoof_ingress",
              "nat_steady_64": "nat44_egress", "nat_cold_64": "nat44_egress", "nat_ingress_64": "nat44_ingress",
              "qos_64": "qos_ingress_prog", "qos_egress_64": "qos_egress_prog", "dhcp": "dhcp_fastpath_prog"}


def workload_config(name: str, frames: int, world: int) -> dict:
    """What the two arms of the bench are run ON — the same dict in the GPU line and in the --impl reference line
    of the same N (everything that describes HOW an arm ran goes under its own "details" key)."""
    return {"workload": name, "program": PROGRAM_OF.get(name, name), "frames_per_gpu_per_step": frames, "gpus": world,
            "subscribers_total": "10 000 (BASELINE config #4), split over the GPUs" if name.startswith("pipeline") else "see bng_b200/workloads.py",
            "sharding": f"splitmix64(mac) % {world}"}


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cpus = host_cpus()
    procs = max(1, min(cpus["usable"], 128))
    n = 1 << 18
    t0 = time.time()
    mpps, kind, tmax = cpu_run(a.workload, n, procs, a.steps, a.warmup)
    out = {
        "impl": "reference", "metric": METRIC, "value": round(mpps, 3), "unit": "Mpps", "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": round(tmax / a.steps * 1e3, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8/u32/u64 integer", "data": "synthetic",
        "config": workload_config(a.workload, a.frames, a.gpus),
        "details": {"frames_per_step_timed": n * procs, "host_procs": procs, "host_cpus": cpus,
                    "state": "subscribers split over the processes by MAC hash, one private map set per process",
                    "note": "a bounded sample of the workload per step (cpu_baseline.sample); under torchrun rank 0 alone runs"},
        "cpu_baseline": {"value": round(mpps, 3), "unit": "Mpps", "cores": procs,
                         "kind": "reference" if kind == "reference" else "port",
                         "sample": f"{procs} processes (sched_getaffinity {cpus['sched_affinity']}, cgroup quota "
                                   f"{cpus['cgroup_quota_cpus']}, os.cpu_count {cpus['os_cpu_count']}) x {n} frames x {a.steps} "
                                   f"steps of {a.workload}; reference eBPF C compiled natively (gcc -O2) over a userspace map runtime"},
        "e2e": {"value": round(mpps, 3), "unit": "Mpps", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": round(time.time() - t0, 1),
    }
    print(json.dumps(out), flush=True)


# ---------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------
def host_arena(nbytes: int):
    """Frame arena for the end-to-end leg from the library's own allocator: bng_host_alloc() = 2 MB transparent
    huge pages registered with CUDA (falls back to cudaHostAlloc).  Returned as a torch uint8 view; arenas live
    until the process ends."""
    import ctypes
    import torch
    from bng_b200.dataplane import load_library
    lib = load_library()
    p = lib.bng_host_alloc(nbytes)
    if not p:
        raise RuntimeError("bng_host_alloc failed")
    arr = np.ctypeslib.as_array((ctypes.c_uint8 * nbytes).from_address(p))
    return torch.from_numpy(arr)


def bind_to_gpu_numa_node(index: int):
    """Pin this process to the CPUs NVML reports as local to GPU `index`, so that first-touch places
    the pinned host buffers on the GPU's NUMA node (PCIe traffic then stays off the socket interconnect)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [64 * w + b for w in range(len(mask)) for b in range(64) if (mask[w] >> b) & 1]
        allowed = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in allowed]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"cpus": f"{cpus[0]}-{cpus[-1]}", "count": len(cpus)}
    except Exception as e:  # affinity is an optimisation, never a requirement
        return {"error": str(e)[:80]}
    return None


class G:
    """Process-wide state of the GPU arm (one rank)."""
    rank = 0
    world = 1
    local = 0
    dev = None
    dist = None
    as_shard = None


def _traffic(name, kernel, world, reference_capacities):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture, with the capture it came from.
    The capture is of ONE configuration (N = 1, workload-sized tables): any other run reports null."""
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(tp) or world != 1 or reference_capacities:
        return None, "not captured for this configuration (profiles/ncu_traffic.json holds the N=1 workload-sized run)"
    ent = json.load(open(tp)).get(name, {}).get(kernel)
    if ent is None:
        return None, "no capture of this kernel"
    if isinstance(ent, dict):
        return ent.get("bytes"), ent.get("source")
    return ent, "profiles/ncu_traffic.json"


# --dump-outputs writes at most 36 + 2 x 12 MiB (under 64 MB).  The frame sample depends on the batch alone, not on
# what a build emitted, so two builds dump the same frames.
DUMP_FRAME_BYTES = 36 << 20  # frames, verdicts, lengths and frame indices
DUMP_EVENT_BYTES = 12 << 20  # records of one event ring


def dump_outputs(out_dir, n, hw, arena_d, off_d, stride, len_d, verdict_d, events):
    """What the last timed step handed back, as DIR/<name>.npy: verdict, len and the first `hw` bytes of every frame
    (the bytes the step restored and the program may rewrite), as float32, and the frames' indices (frame_index,
    float64); above DUMP_FRAME_BYTES a fixed seeded sample of frames (sorted) stands for the batch.  And the records
    the step emitted into each event ring (`events`: ring -> u8[records, size], drained after the step), as float32
    bytes with the padding the reference leaves uninitialised zeroed (ev_<ring>: the first DUMP_EVENT_BYTES of them in
    ring order; no file for a ring the step left empty)."""
    import torch
    from bng_b200.layouts import PADDING
    outs = {}
    for ring, rec in events.items():
        if rec.shape[0] == 0:
            continue
        rec = rec[: DUMP_EVENT_BYTES // (4 * rec.shape[1])].copy()
        for off, ln in PADDING.get(ring, ()):
            rec[:, off:off + ln] = 0
        outs["ev_" + ring] = rec.astype(np.float32)
    per_frame = (hw + 2) * 4 + 8
    if n * per_frame <= DUMP_FRAME_BYTES:
        idx = np.arange(n, dtype=np.int64)
    else:
        idx = np.sort(np.random.default_rng(0xB200).choice(n, DUMP_FRAME_BYTES // per_frame, replace=False))
    idx_d = torch.from_numpy(idx).to(arena_d.device)
    if off_d is None:
        frames = arena_d[: n * stride].view(n, stride)[idx_d, :hw]
    else:
        frames = arena_d[off_d.long()[idx_d, None] * 16 + torch.arange(hw, device=arena_d.device)[None, :]]
    os.makedirs(out_dir, exist_ok=True)
    outs.update({"frame_index": idx.astype(np.float64), "verdict": verdict_d[idx_d].cpu().numpy().astype(np.float32),
                 "len": len_d[idx_d].cpu().numpy().astype(np.float32), "frames": frames.cpu().numpy().astype(np.float32)})
    for k, v in outs.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def measure(a, name, frames, steps, warmup, *, wl=None, reference_capacities=False, subs_scale=1, keep=False, dump=None):
    """One workload on this rank's GPU: W warm-up steps, K timed steps (CUDA events on the library's stream, fresh
    frames restored untimed between steps), max over ranks, then a per-kernel pass for the roofline.  Returns the
    result dict; with keep=True also the live objects the end-to-end leg needs; with dump=DIR the outputs of the last
    timed step are written there (dump_outputs)."""
    import torch
    from bng_b200 import MEM_DEVICE, Dataplane
    from bng_b200.layouts import as_bytes
    dev, dist, world, rank = G.dev, G.dist, G.world, G.rank
    if wl is None:
        wl = W.build(name, frames, *(G.as_shard or (rank, world)), subs_scale)
    n = wl.n
    sr, sw = G.as_shard or (rank, world)
    dp = Dataplane(device=G.local, max_batch=max(n, 1 << 20), rank=sr, world=sw,
                   **({} if reference_capacities else W.sizing(wl)))
    for m, k, v in wl.maps:
        r = dp.update_batch(m, as_bytes(k), as_bytes(v))
        assert r == 0, (m, r)
    translated = []
    for prog, h, l in wl.prewarm:  # e.g. create the NAT sessions of every flow once (cold start), untimed
        ph = torch.from_numpy(h).to(dev).reshape(-1)
        pl = torch.from_numpy(l.astype(np.int32)).to(dev)
        torch.cuda.synchronize()
        dp.run(prog, ph, pl, wl.now0 - 1, stride=64, mem=MEM_DEVICE)
        dp.sync()
        if wl.derive is not None:
            translated.append(ph.cpu().numpy())
    if wl.derive is not None and not getattr(wl, "_derived", False):
        wl.headers, wl.lens = wl.derive(translated)
        wl._derived = True
    hw = wl.headers.shape[1]
    off16, stride, total16 = W.slot16(wl.lens, wl.imix, hw, a.align)
    hdr_d = torch.from_numpy(wl.headers).to(dev)
    len0_d = torch.from_numpy(wl.lens.astype(np.int32)).to(dev)
    len_d = len0_d.clone()
    arena_d = torch.zeros(total16 * 16 + 64, dtype=torch.uint8, device=dev)
    a16 = arena_d[: total16 * 16].view(total16, 16)
    off_d = gidx = None
    if off16 is not None:
        off_d = torch.from_numpy(off16.astype(np.int32)).to(dev)
        gidx = off_d.long()[:, None] + torch.arange(hw // 16, device=dev)[None, :]
    verdict_d = torch.zeros(n, dtype=torch.uint8, device=dev)
    lib_stream = torch.cuda.ExternalStream(dp.stream, device=dev)

    def reset_state():
        for ring in ("spoof_events", "nat_log_rb"):  # the event consumer keeps the staging rings empty (untimed)
            dp.drain(ring)
        if wl.name == "nat_cold_64":  # every step starts from empty flow tables and fresh port blocks
            for m in ("nat_sessions", "nat_reverse", "eim_table"):
                dp.clear(m)
            for m, k, v in wl.maps:
                if m == "subscriber_nat":
                    dp.update_batch(m, as_bytes(k), as_bytes(v))

    def restore():
        dp.sync()  # the previous step (asynchronous on the library's stream) must be done with the arena
        if off16 is None:
            arena_d[: n * stride].view(n, stride)[:, :hw] = hdr_d
        else:
            a16[gidx.reshape(-1)] = hdr_d.view(-1, 16)
        len_d.copy_(len0_d)
        torch.cuda.synchronize()
        reset_state()

    step_no = [0]

    def step():
        now = wl.now0 + step_no[0] * wl.now_step
        step_no[0] += 1
        dp.run(wl.prog, arena_d, len_d, now, off16=off_d, stride=stride, verdict=verdict_d, mem=MEM_DEVICE)

    for _ in range(warmup):
        restore()
        step()
        dp.sync()
    sampler = ClockSampler(G.local)
    sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches0 = dp.launch_count
    evs = []
    for _ in range(steps):
        restore()  # fresh frames for this step (untimed: stands in for the NIC filling the arena)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(lib_stream)
        step()
        e1.record(lib_stream)
        evs.append((e0, e1))
    dp.sync()
    torch.cuda.synchronize()
    launches = dp.launch_count - launches0
    step_ms = [e0.elapsed_time(e1) for e0, e1 in evs]
    tmax = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    nsum = torch.tensor([n], dtype=torch.float64, device=dev)
    if world > 1:
        dist.barrier()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(nsum, op=dist.ReduceOp.SUM)
    total_ms_max = float(tmax.item())
    frames_all = float(nsum.item())
    clocks = sampler.result()
    drops = int((verdict_d == 2).sum().item())
    value = frames_all * steps / (total_ms_max * 1e-3) / 1e6
    if dump:  # before the per-kernel pass below overwrites the arena
        dump_outputs(dump, n, hw, arena_d, off_d, stride, len_d, verdict_d,
                     {ring: dp.drain(ring) for ring in ("spoof_events", "nat_log_rb")})

    # ---- per-kernel timing for the roofline (separate pass, events around every launch) ----
    dp.prof_enable(True)
    for _ in range(3):
        restore()
        step()
        dp.sync()
    prof = dp.prof_read()
    dp.prof_enable(False)
    top = max(prof.items(), key=lambda kv: kv[1][1])
    top_ms = top[1][1] / top[1][0]
    step_prof_ms = sum(v[1] for v in prof.values()) / 3
    peak, peak_src = peaks()
    algo = W.ALGO_BYTES[wl.name]
    traffic, traffic_src = _traffic(wl.name, top[0], world, reference_capacities)
    achieved = algo * n / (top_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": top[0], "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_frame": algo, "kernel_ms": round(top_ms, 4),
                "kernel_share_of_step": round(top[1][1] / 3 / step_prof_ms, 3),
                "step_frac": round(algo * n / (total_ms_max / steps * 1e-3) / 1e9 / peak, 4),
                "kernels_ms": {k: round(v[1] / v[0], 4) for k, v in prof.items()}}
    res = {"value": round(value, 2), "unit": "Mpps", "ms_per_step": round(total_ms_max / steps, 4), "steps": steps, "warmup": warmup,
           "frames_per_gpu_per_step": n, "subscribers_this_gpu": wl.n_subs_local, "step_ms": [round(float(x), 3) for x in step_ms],
           "roofline": roofline, "gpu_launches": int(launches), "clocks": clocks, "drop_fraction_last_step": round(drops / n, 4),
           "tables": "reference capacities (1 M subscribers, 4 M sessions, 2 M EIM)" if reference_capacities else
                     "sized for the provisioned subscribers / flows (2x head-room)",
           "lru_overflow": int(dp.lru_overflow), "events_lost": int(dp.events_lost)}
    if keep:
        live = dict(dp=dp, wl=wl, off16=off16, stride=stride, total16=total16, hw=hw, gidx=gidx, step_no=step_no,
                    reset_state=reset_state, n=n, arena_bytes=total16 * 16)
        return res, live
    dp.close()
    del arena_d, hdr_d
    torch.cuda.empty_cache()
    return res, None


def e2e_leg(a, live):
    """The same metric through bng_prog_run(BNG_MEM_HOST): frames in a pinned host arena, host<->device copies inside
    the timed region (wall clock around the call, max over ranks)."""
    import torch
    from bng_b200 import MEM_HOST
    dev, dist, world = G.dev, G.dist, G.world
    dp, wl, off16, stride, total16, hw, gidx = (live[k] for k in ("dp", "wl", "off16", "stride", "total16", "hw", "gidx"))
    n, step_no, reset_state = live["n"], live["step_no"], live["reset_state"]
    e2e_steps = max(1, min(a.steps, a.e2e_steps))
    n_e = min(n, max(1, a.e2e_frames))
    lens_e, hdrs_e = wl.lens[:n_e], wl.headers[:n_e]
    off16_e = off16[:n_e] if off16 is not None else None
    total16_e = total16 if n_e == n else (int(off16[n_e]) if off16 is not None else n_e * stride // 16)
    arena_h = host_arena(total16_e * 16 + 64)

    def host_like(t):
        h = host_arena(t.numel() * t.element_size()).view(t.dtype)[: t.numel()]
        h.copy_(t)
        return h

    len_h = host_like(torch.from_numpy(lens_e.astype(np.int32)))
    off_h = host_like(torch.from_numpy(off16_e.astype(np.int32))) if off16 is not None else None
    verdict_h = host_like(torch.zeros(n_e, dtype=torch.uint8))
    hdr_h = torch.from_numpy(np.ascontiguousarray(hdrs_e))
    len0_h = torch.from_numpy(lens_e.astype(np.int32))
    h16 = arena_h[: total16_e * 16].view(total16_e, 16)
    gidx_h = gidx[:n_e].reshape(-1).cpu() if off16 is not None else None

    def restore_host():
        if off16 is None:
            arena_h[: n_e * stride].view(n_e, stride)[:, :hw] = hdr_h
        else:
            h16.index_copy_(0, gidx_h, hdr_h.view(-1, 16))
        len_h.copy_(len0_h)

    tc_prog = wl.prog != "dhcp_fastpath_prog"
    hb = 64 if tc_prog else 448  # bytes of each frame that cross PCIe from a pinned arena (96 when ihl > 5)

    def run(arena_t, off_t, strd, restore_fn, nbytes):
        tot = 0.0
        for s in range(1 + e2e_steps):
            restore_fn()
            reset_state()
            dp.sync()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            now = wl.now0 + step_no[0] * wl.now_step
            step_no[0] += 1
            dp.run(wl.prog, arena_t, len_h, now, off16=off_t, stride=strd, verdict=verdict_h, mem=MEM_HOST, arena_bytes=nbytes)
            dt = time.perf_counter() - t0
            if s >= 1:
                tot += dt
        et = torch.tensor([tot], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(et, op=dist.ReduceOp.MAX)
        return world * n_e * e2e_steps / float(et.item()) / 1e6

    val = run(arena_h, off_h, stride, restore_host, total16_e * 16)
    per_frame_in = float(np.minimum(lens_e, hb).mean())
    h2d = int(n_e * per_frame_in) + n_e * 4 + (n_e * 4 if off16 is not None else 0)
    d2h = int(n_e * per_frame_in) + n_e + (n_e * 4 if not tc_prog else 0)  # (whole 64-byte header slots go back: one write per frame)
    out = {"value": round(val, 2), "unit": "Mpps", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
           "steps": e2e_steps, "frames_per_step": n_e, "arena": "bng_host_alloc(): 2 MB huge pages registered with CUDA",
           "layout": "pinned host arena, full frames; only the bytes a program can touch cross PCIe"}
    extra = None
    if tc_prog and wl.imix:
        # header-split receive: the NIC put the first 64 bytes of every frame in a contiguous ring (len[] still
        # carries the full frame length, bounds checks stop at the slot: tests/test_gpu_slots.py)
        ring_h = host_arena(n_e * 64)

        def restore_ring():
            ring_h.view(n_e, 64)[:, :hw] = hdr_h
            len_h.copy_(len0_h)

        v = run(ring_h, None, 64, restore_ring, n_e * 64)
        extra = {"value": round(v, 2), "unit": "Mpps", "layout": "header-split ring (64 B per frame, len = full frame)",
                 "h2d_bytes_per_step": n_e * 64 + n_e * 4, "d2h_bytes_per_step": n_e * 64 + n_e}
    return out, extra


EXTRA_WORKLOADS = ("antispoof_64", "nat_steady_64", "nat_cold_64", "dhcp")


def control_plane_leg(dp, wl):
    """What the Go side does between batches, timed on the live context of the headline run (host clock around the
    C-ABI calls, which are synchronous): one Map.Put (bng_map_update), staged upserts applied at the next batch
    boundary (bng_map_update_staged + bng_sync), a batch upsert, and the expiry sweep over the live nat_sessions
    table (one streaming pass: 64 of every slot's 128 bytes).  Not part of the headline metric."""
    from bng_b200.layouts import as_bytes
    out = {}
    qm = [(m, k, v) for m, k, v in wl.maps if m == "qos_ingress"]
    if qm:
        _, k, v = qm[0]
        kb, vb = as_bytes(k), as_bytes(v)
        m = min(len(kb), 20000)
        t = []
        for i in range(min(m, 300)):
            t0 = time.perf_counter()
            dp.update("qos_ingress", kb[i], vb[i])
            t.append(time.perf_counter() - t0)
        out["put_single_us"] = {"median": round(float(np.median(t)) * 1e6, 1), "p99": round(float(np.percentile(t, 99)) * 1e6, 1),
                                "n": len(t), "what": "bng_map_update(qos_ingress), synchronous, through ctypes"}
        t0 = time.perf_counter()
        for i in range(m):
            dp.update_staged("qos_ingress", kb[i], vb[i])
        t1 = time.perf_counter()
        dp.sync()
        t2 = time.perf_counter()
        out["put_staged"] = {"n": m, "stage_us_each": round((t1 - t0) / m * 1e6, 2), "apply_ms": round((t2 - t1) * 1e3, 3),
                             "puts_per_s": round(m / (t2 - t0)), "what": "bng_map_update_staged x n, applied by one bng_sync"}
        t0 = time.perf_counter()
        dp.update_batch("qos_ingress", kb[:m], vb[:m])
        dt = time.perf_counter() - t0
        out["put_batch"] = {"n": m, "ms": round(dt * 1e3, 3), "puts_per_s": round(m / dt)}
    info = dp.map_info("nat_sessions")
    live = info["count"]
    if live:
        slots = 1
        while slots < 2 * info["max_entries"]:
            slots *= 2
        dp.sync()
        t0 = time.perf_counter()
        expired = dp.sweep(wl.now0 + 300 * 10**9)
        dt = time.perf_counter() - t0
        t0 = time.perf_counter()
        dp.sweep(wl.now0 + 300 * 10**9)  # second pass: nothing left to expire = the pure scan
        dt2 = time.perf_counter() - t0
        out["sweep"] = {"live_sessions": int(live), "slots": slots, "expired": int(expired), "ms": round(dt * 1e3, 3),
                        "scan_only_ms": round(dt2 * 1e3, 3), "scan_GBps": round(slots * 64 / dt2 / 1e9, 1),
                        "table_rebuilds": int(dp.table_rebuilds),
                        "what": "bng_sweep at now + 300 s (UDP, ICMP and non-established TCP flows expire); host clock, "
                                "includes the launch + sync; scan bytes = 64 per 128-byte slot"}
    return out


def run_gpu(a):
    import torch
    import torch.distributed as dist
    from bng_b200 import Dataplane

    G.rank = rank = int(os.environ.get("RANK", "0"))
    G.world = world = int(os.environ.get("WORLD_SIZE", "1"))
    G.local = local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly one JSON line: whatever native libraries print there while we run (NCCL's version
    # banner, for one) goes to stderr instead
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    numa = bind_to_gpu_numa_node(local)  # pinned host buffers must live next to the GPU's PCIe root
    # The untimed host-side refills of the frame arena are torch copies that fan out over every CPU the process can
    # see (64+); under a cgroup CPU quota (16 on the 1-GPU boxes) such a burst spends the whole period's allowance and
    # the kernel then freezes the cgroup for the rest of the period — right when the timed bng_prog_run call runs
    # (tools/e2e_diag.py: one 50 ms step among 2.4 ms ones).  Stay well inside the quota.
    hc = host_cpus()
    torch.set_num_threads(max(1, min(8, hc["usable"] // 2)))
    torch.cuda.set_device(local)
    G.dev = dev = torch.device("cuda", local)
    G.dist = dist
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    t_start = time.time()

    # ---- headline: the workload at BASELINE's population, tables sized for it ----
    dump = a.dump_outputs and (a.dump_outputs if world == 1 else os.path.join(a.dump_outputs, f"rank{rank}"))
    head, live = measure(a, a.workload, a.frames, a.steps, a.warmup, reference_capacities=a.reference_capacities, keep=True,
                         dump=dump)
    wl, dp = live["wl"], live["dp"]
    e2e, e2e_extra = e2e_leg(a, live) if a.e2e_steps > 0 else (None, None)  # 0: kernel-only runs under a profiler

    # ---- counter reconciliation: NCCL all-reduce of the packed counter vector INSIDE the library (bng_sync_reduce)
    #      over a communicator of the library's own; the unique id travels through the host plumbing ----
    uid = [Dataplane.comm_unique_id() if rank == 0 else None]
    if world > 1:
        dist.broadcast_object_list(uid, src=0)
    t0 = time.perf_counter()
    dp.comm_init(uid[0], rank, world)
    t_comm = time.perf_counter() - t0
    dp.sync_reduce()  # first collective on a new communicator sets up its channels: untimed
    t0 = time.perf_counter()
    stats_global = dp.sync_reduce()
    t_red = time.perf_counter() - t0
    ptr, nst = dp.stats_device_ptr()
    mine = torch.as_tensor(DevPtr(ptr, nst), device=dev).clone()
    check = mine.clone()
    if world > 1:
        dist.all_reduce(check, op=dist.ReduceOp.SUM)  # the same reduction by torch: must agree
    reduce_ok = bool((check.cpu().numpy().view(np.uint64) == stats_global).all())
    coop = (int(mine[37].item()), int(mine[38].item()))
    ctl = control_plane_leg(dp, wl) if rank == 0 and not a.no_extra else None
    dp.close()
    del live
    torch.cuda.empty_cache()

    # ---- the same workload with every table at the reference's compile-time capacity ----
    refcap = None
    if not a.reference_capacities and not a.no_extra:
        r, _ = measure(a, a.workload, a.frames, max(3, min(a.steps, 10)), 3, wl=wl, reference_capacities=True)
        refcap = {k: r[k] for k in ("value", "unit", "ms_per_step", "tables")}
        refcap["roofline"] = {k: r["roofline"][k] for k in ("kernel", "kernel_ms", "frac", "step_frac", "kernels_ms")}
    # ---- 10 k subscribers PER GPU (population grows with N: per-GPU tables keep their size) ----
    pergpu = None
    if not a.no_extra:
        if world == 1:
            pergpu = {"value": head["value"], "ms_per_step": head["ms_per_step"], "note": "identical to the headline at N = 1"}
        else:
            r, _ = measure(a, a.workload, a.frames, max(3, min(a.steps, 10)), 3, subs_scale=world)
            pergpu = {k: r[k] for k in ("value", "unit", "ms_per_step", "subscribers_this_gpu", "drop_fraction_last_step")}
            pergpu["roofline"] = {k: r["roofline"][k] for k in ("kernel", "kernel_ms", "frac", "step_frac", "kernels_ms")}
    # ---- the other BASELINE configs, short (5 steps), sharded the same way ----
    others = {}
    if not a.no_extra:
        for name in EXTRA_WORKLOADS:
            if name == a.workload:
                continue
            r, _ = measure(a, name, a.frames, 5, 3)
            rf = r["roofline"]
            others[name] = {"value": r["value"], "unit": "Mpps", "ms_per_step": r["ms_per_step"], "kernel": rf["kernel"],
                            "kernel_ms": rf["kernel_ms"], "frac": rf["frac"], "step_frac": rf["step_frac"], "traffic": rf["traffic"],
                            "traffic_source": rf["traffic_source"], "algorithmic_bytes_per_frame": rf["algorithmic_bytes_per_frame"],
                            "kernels_ms": rf["kernels_ms"], "frames_per_gpu_per_step": r["frames_per_gpu_per_step"],
                            "subscribers_this_gpu": r["subscribers_this_gpu"], "gpu_launches": r["gpu_launches"]}

    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu:
        c_n = 1 << 20
        mpps, kind, tt = cpu_run(a.workload, c_n, 1, 20, 1)  # ~10 s of one core
        cpu = {"value": round(mpps, 3), "unit": "Mpps", "cores": 1, "kind": kind,
               "sample": f"1 core x {c_n} frames x 20 passes of {a.workload} ({tt:.1f} s), reference eBPF C run natively"}
    if rank == 0:
        out = {
            "metric": METRIC, "value": head["value"], "unit": "Mpps", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8/u32/u64 integer", "data": "synthetic",
            "config": workload_config(wl.name, head["frames_per_gpu_per_step"], world),
            "details": {"frames_this_gpu": head["frames_per_gpu_per_step"], "subscribers_this_gpu": wl.n_subs_local,
                        "sharding": f"splitmix64(mac) % {world}" if not G.as_shard else f"diagnostic: shard {G.as_shard[0]} of {G.as_shard[1]} alone",
                        "tables": head["tables"], "avg_frame_bytes": round(float(wl.lens.mean()), 1),
                        "frame_align": a.align if wl.imix else live_stride(wl),
                        "step_ms_min_med_max": [round(float(x), 4) for x in
                                                (min(head["step_ms"]), float(np.median(head["step_ms"])), max(head["step_ms"]))],
                        "step_ms_all": head["step_ms"],
                        "l2_policy": "inputs larger than L2 (frame arena + tables) and rewritten between steps",
                        **wl.info},
            "wire_gbps": round(head["value"] * 1e6 * float(wl.lens.mean()) * 8 / 1e9, 1),
            "roofline": head["roofline"], "cpu_baseline": cpu,
            "e2e": e2e, "e2e_header_split": e2e_extra, "host_affinity": numa,
            "gpu_launches": head["gpu_launches"], "clocks": head["clocks"],
            "verdict_drop_fraction_last_step": head["drop_fraction_last_step"],
            "reference_capacities": refcap, "per_gpu_constant": pergpu, "workloads": others,
            "stats_allreduce": {"by": "bng_sync_reduce (ncclAllReduce inside libbng_b200.so)", "matches_torch_allreduce": reduce_ok,
                                "comm_init_s": round(t_comm, 3), "reduce_ms": round(t_red * 1e3, 3),
                                "antispoof_allowed": int(stats_global[0]), "nat_snat": int(stats_global[10]),
                                "qos_dropped": int(stats_global[7])},
            "lru_overflow": head["lru_overflow"], "events_lost": head["events_lost"],
            "control_plane": ctl,
            "nat_ordered_frames": {"cooperative": coop[0], "sequential": coop[1]},
            "wall_s": round(time.time() - t_start, 1),
        }
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(out) + "\n").encode())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def live_stride(wl):
    return ((wl.headers.shape[1] + 15) // 16) * 16


class DevPtr:
    """__cuda_array_interface__ wrapper so torch can view library-owned device memory."""

    def __init__(self, ptr, n, typestr="<i8"):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}


def run_dhcp_slow(a):
    """BASELINE.json configs[0]: 1 000 DHCP DISCOVERs through the slow path with a 256-entry lease map, CPU only.
    The reference's pkg/dhcp is Go and cannot be built in this image; what is timed is its C++ restatement
    (bng_b200/host/bng_dhcp_slow.hpp, one thread — the reference serialises on the pool mutex).  Plumbing: no GPU,
    no roofline, gpu_launches 0 by construction."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_host_mirror
    test_host_mirror.build_host_test()
    rounds = a.steps  # one step = one round of 1 000 DISCOVERs
    j = json.loads(subprocess.run([test_host_mirror.SLOW_BIN, str(rounds)], capture_output=True, text=True, check=True).stdout)
    print(json.dumps({
        "metric": "DHCP DISCOVER/s (slow path, CPU only)", "value": round(j["req_per_s"], 1), "unit": "requests/s", "n_gpus": 0,
        "steps": rounds, "warmup": 0, "ms_per_step": round(j["seconds"] / rounds * 1e3, 4), "higher_is_better": True,
        "scaling": "n/a", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "dhcp_slow", "requests_per_step": 1000, "clients_with_lease": 256, "pool": "10.0.0.0/22",
                   "implementation": "C++ restatement of pkg/dhcp Server.handleDiscover + Pool.Allocate (Go toolchain absent)"},
        "roofline": None, "gpu_launches": 0,
        "cpu_baseline": {"value": round(j["req_per_s"], 1), "unit": "requests/s", "cores": 1, "kind": "port",
                         "sample": f"{j['requests']} DISCOVERs in {j['seconds']:.2f} s"},
        "e2e": {"value": round(j["req_per_s"], 1), "unit": "requests/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "replies_fnv1a": j["replies_fnv1a"]}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of the headline, of --impl reference and of dhcp_slow (1 000 DISCOVERs each).  The "
                         "side measurements of the GPU arm keep their own counts: the end-to-end leg min(K, --e2e-steps), "
                         "the reference-capacities and per-GPU-constant variants min(max(K, 3), 10), the other "
                         "workloads 5, the one-core CPU baseline 20 passes")
    ap.add_argument("--warmup", type=int, default=3, help="untimed steps before the timed ones (at least 3 on the GPU)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="pipeline_imix", choices=sorted(W.BUILDERS) + ["dhcp_slow"],
                    help="dhcp_slow = BASELINE config #1: the DHCP slow path (CPU only, plumbing; no GPU involved)")
    ap.add_argument("--frames", type=int, default=1 << 22)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--e2e-frames", type=int, default=1 << 20, help="frames per bng_prog_run call in the end-to-end leg")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--reference-capacities", action="store_true",
                    help="size every table for the reference's compile-time max_entries instead of the workload")
    ap.add_argument("--align", type=int, default=64, help="frame placement granularity in the IMIX arena (16 or 64)")
    ap.add_argument("--as-shard", default=None, metavar="R/N",
                    help="diagnostic: run ONE GPU as shard R of an N-GPU job (its subscribers, its frames) without the other ranks")
    ap.add_argument("--no-extra", action="store_true",
                    help="only the headline: skip the reference-capacities variant, the per-GPU-constant variant and the other configs")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the headline's last timed step computed (verdicts, lengths, frame bytes, event "
                         "records; a fixed sample of frames above 36 MiB) to DIR/<name>.npy as float32, to "
                         "compare two builds")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "ours" or a.workload == "dhcp_slow"):
        ap.error("--dump-outputs writes the outputs of the GPU arm")
    a.warmup = max(a.warmup, 3) if a.impl == "ours" else a.warmup
    if a.as_shard:
        G.as_shard = tuple(int(x) for x in a.as_shard.split("/"))
    if a.workload == "dhcp_slow":
        run_dhcp_slow(a)
    elif a.impl == "reference":
        run_reference_arm(a)
    else:
        run_gpu(a)


if __name__ == "__main__":
    main()
