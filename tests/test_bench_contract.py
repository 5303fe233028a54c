"""bench.py's JSON-line contract for the arms that need no GPU: the reference arm (the reference's eBPF C on the host
cores) and BASELINE config #1 (DHCP slow path); on the GPU, the outputs --dump-outputs writes.  One line on stdout,
the keys a consumer of the line reads."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import pyoracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
            "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"]


def run_bench(*args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout  # exactly one line, and it is the JSON
    return json.loads(lines[0])


@pytest.mark.skipif(not (pyoracle.available("reference") or pyoracle.available("port")), reason="no oracle library built")
@pytest.mark.parametrize("workload", ["antispoof_64", "nat_ingress_64"])
def test_reference_arm_line(workload):
    j = run_bench("--impl", "reference", "--workload", workload, "--steps", "1", "--warmup", "0")
    for k in REQUIRED:
        assert k in j, k
    assert j["impl"] == "reference" and j["value"] > 0 and j["unit"] == "Mpps"
    assert j["config"]["workload"] == workload
    # both arms describe WHAT they ran with the same dict (the driver compares them); how an arm ran is under "details"
    sys.path.insert(0, ROOT)
    import bench
    assert j["config"] == bench.workload_config(workload, 1 << 22, 1) and "host_procs" in j["details"]
    assert j["cpu_baseline"]["kind"] in ("reference", "port") and j["cpu_baseline"]["cores"] >= 1
    assert j["e2e"]["value"] == j["value"] and j["e2e"]["h2d_bytes_per_step"] == 0 and j["gpu_launches"] == 0


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_config1_dhcp_slow_line():
    j = run_bench("--workload", "dhcp_slow", "--steps", "1")
    for k in REQUIRED:
        assert k in j, k
    assert j["n_gpus"] == 0 and j["gpu_launches"] == 0 and j["roofline"] is None
    assert j["unit"] == "requests/s" and j["value"] > 1e4 and j["steps"] == 1
    assert j["config"]["clients_with_lease"] == 256 and j["config"]["requests_per_step"] == 1000


@pytest.mark.gpu
@pytest.mark.parametrize("workload,n", [("pipeline_imix", 1 << 15), ("pipeline_64", 1 << 22)])
def test_dump_outputs_are_the_last_timed_step(tmp_path, workload, n):
    """--steps K times K steps, and --dump-outputs writes what the last of them computed: the same verdicts, lengths,
    frame bytes and event records as the oracle after warm-up + K passes over the same workload.  2^15 IMIX frames sit
    in a packed arena and are dumped whole; 2^22 64-byte frames sit at a fixed stride and only a sample fits."""
    from bng_b200 import layouts as L
    from bng_b200 import workloads as W
    from bng_b200.layouts import as_bytes
    sys.path.insert(0, ROOT)
    import bench
    warmup, steps = 3, 2
    j = run_bench("--workload", workload, "--frames", str(n), "--steps", str(steps), "--warmup", str(warmup),
                  "--no-extra", "--no-cpu", "--e2e-steps", "0", "--dump-outputs", str(tmp_path))
    assert j["steps"] == steps and len(j["details"]["step_ms_all"]) == steps
    rings = ("spoof_events", "nat_log_rb")
    got = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert {"frame_index", "verdict", "len", "frames"} <= set(got) <= {"frame_index", "verdict", "len", "frames"} | {
        "ev_" + r for r in rings}
    assert all(v.dtype in (np.float32, np.float64) and v.size > 0 for v in got.values())
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= 64_000_000
    idx = got["frame_index"].astype(np.int64)
    assert np.array_equal(got["frame_index"], idx) and (np.diff(idx) > 0).all() and 0 <= idx[0] and idx[-1] < n
    per_frame = (64 + 2) * 4 + 8  # float32 header bytes, verdict and len, float64 index
    assert len(idx) == (n if n * per_frame <= bench.DUMP_FRAME_BYTES else bench.DUMP_FRAME_BYTES // per_frame)

    wl = W.BUILDERS[workload](n, 0, 1)
    o = pyoracle.Oracle("port")
    for m, k, v in wl.maps:
        o.update_batch(m, as_bytes(k), as_bytes(v))
    for prog, h, l in wl.prewarm:
        pa = o.arena(h.shape[0] * 64 + 64)
        pa[: h.shape[0] * 64] = h.reshape(-1)
        o.run(prog, pa, l.copy(), wl.now0 - 1, stride=64)
    hw = wl.headers.shape[1]
    off16, stride, total16 = W.slot16(wl.lens, wl.imix, hw)
    arena = o.arena(total16 * 16 + 64)
    if off16 is None:
        view = arena[: n * stride].reshape(n, stride)
    else:
        pos = off16.astype(np.int64)[:, None] * 16 + np.arange(hw)[None, :]
    for s in range(warmup + steps):
        if off16 is None:
            view[:, :hw] = wl.headers
        else:
            arena[pos] = wl.headers
        lens = wl.lens.copy()
        verdict = o.run(wl.prog, arena, lens, wl.now0 + s * wl.now_step, off16=off16, stride=stride)
        events = {r: o.drain(r) for r in rings}  # what this step emitted
    frames = view[idx, :hw] if off16 is None else arena[pos[idx]]
    assert np.array_equal(got["verdict"], verdict[idx].astype(np.float32))
    assert np.array_equal(got["len"], lens[idx].astype(np.float32))
    assert np.array_equal(got["frames"], frames.astype(np.float32))
    assert events["spoof_events"].shape[0] > 0
    for r in rings:
        if events[r].shape[0] == 0:  # (nat_log_rb: these workloads create their sessions in the untimed prewarm)
            assert "ev_" + r not in got, r
            continue
        want = events[r][: bench.DUMP_EVENT_BYTES // (4 * events[r].shape[1])].copy()
        for off, ln in L.PADDING.get(r, ()):
            want[:, off:off + ln] = 0
        assert np.array_equal(got["ev_" + r], want.astype(np.float32)), r
