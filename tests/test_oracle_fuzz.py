"""Mutation fuzzing of the parsers: valid frames of the scenario corpora are truncated, bit-flipped and given odd
header lengths / ethertypes, then run through the plain-C port with the scenario's map contents and compared with
the reference's C: with the fingerprints of its results (tests/golden/mutated_frames.json, written by
tests/golden/make_golden.py) and, where the reference build (oracle/_ref) is present, with a live run.  Everything
observable must agree bit for bit.  This is where bounds checks live (frames shorter than a header, ihl != 5, VLAN
tags, option walks running off the end), i.e. where a restatement is most likely to drift from the original."""
import json
import os

import numpy as np
import pytest

import harness
import scenarios
from harness import Script
from oracle import pyoracle

SEEDS = [11, 12]
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mutated_frames.json")

TARGETS = {  # program -> (scenario providing maps + seed frames, index of the run step to take frames from)
    "antispoof_ingress": "antispoof",
    "qos_ingress_prog": "qos",
    "qos_egress_prog": "qos",
    "nat44_egress": "nat",
    "nat44_ingress": "nat",
    "nat44_hairpin_xdp": "nat",
    "pipeline_up": "pipeline",
    "pipeline_tc": "pipeline",
    "dhcp_fastpath_prog": "dhcp",
}


def mutate(frames: np.ndarray, lens: np.ndarray, seed: int, width: int):
    """frames u8[n, width] (fixed slots), lens u32[n] -> mutated copies."""
    r = np.random.Generator(np.random.PCG64(seed))
    f = frames.copy()
    l = lens.copy()
    n = f.shape[0]
    kind = r.integers(0, 10, n)
    # truncate to a random length (including 0..13: shorter than an Ethernet header)
    t = kind == 0
    l[t] = r.integers(0, np.maximum(l[t], 1) + 1)
    t = kind == 1
    l[t] = r.choice(np.array([13, 14, 20, 33, 34, 37, 38, 41, 42, 53, 54], dtype=np.uint32), t.sum())
    # flip a random bit somewhere in the headers (DHCP: anywhere up to the options)
    t = np.nonzero(kind == 2)[0]
    span = min(64, width) if width <= 64 else min(width, 320)
    f[t, r.integers(0, span, len(t))] ^= (1 << r.integers(0, 8, len(t))).astype(np.uint8)
    # (DHCP) garbage over the first option bytes: option walks must stay in bounds
    t = np.nonzero(kind == 7)[0]
    if width > 300:
        f[t, 282:300] = r.integers(0, 256, (len(t), 18), dtype=np.uint8)
    # odd IP header lengths / versions
    t = kind == 3
    f[t, 14] = (f[t, 14] & 0xF0) | r.integers(0, 16, t.sum()).astype(np.uint8)
    # other ethertypes: IPv6, ARP, 802.1Q, 802.1ad, junk
    t = np.nonzero(kind == 4)[0]
    et = r.choice(np.array([0x86DD, 0x0806, 0x8100, 0x88A8, 0x1234], dtype=np.uint32), len(t))
    f[t, 12], f[t, 13] = (et >> 8).astype(np.uint8), (et & 0xFF).astype(np.uint8)
    # other L4 protocols
    t = kind == 5
    f[t, 23] = r.choice(np.array([1, 6, 17, 47, 50, 132, 0], dtype=np.uint8), t.sum())
    # random garbage over the L4 area
    t = np.nonzero(kind == 6)[0]
    if width >= 64:
        f[t, 34:64] = r.integers(0, 256, (len(t), 30), dtype=np.uint8)
    # lengths longer than the slot are not representable in a fixed arena: cap
    l = np.minimum(l, width).astype(np.uint32)
    return f, l


def base_maps_and_frames(scenario: str):
    sc = scenarios.ALL_SCRIPTS[scenario]()
    updates = [st for st in sc.steps if st[0] == "update"]
    run = next(st for st in sc.steps if st[0] == "run")
    _, _, arena, lens, now, off16, stride, _, _ = run
    if off16 is None:
        frames = arena.reshape(-1, stride)[: len(lens)]
        return updates, frames, lens, now, stride
    width = (int(lens.max()) + 31) // 16 * 16  # variable-length corpus (DHCP): repack into fixed slots
    frames = np.zeros((len(lens), width), np.uint8)
    for i, (o, n) in enumerate(zip(off16.astype(np.int64) * 16, lens)):
        frames[i, :n] = arena[o:o + n]
    return updates, frames, lens, now, width


def fuzz_script(prog, seed):
    updates, frames, lens, now, stride = base_maps_and_frames(TARGETS[prog])
    f, l = mutate(frames, lens, seed * 7919 + len(prog), stride)
    sc = Script(f"fuzz_{prog}_{seed}")
    sc.steps = list(updates)
    sc.run(prog, f.reshape(-1).copy(), l.copy(), now + 5, stride=stride)
    sc.run(prog, f[::-1].reshape(-1).copy(), l[::-1].copy(), now + 10 ** 9, stride=stride)  # and again, reversed order
    return sc


@pytest.mark.parametrize("seed", SEEDS)
@pytest.mark.parametrize("prog", sorted(TARGETS))
def test_mutated_frames_agree(prog, seed):
    port = harness.run_script(harness.OracleBackend("port"), fuzz_script(prog, seed))
    with open(GOLD) as f:
        want = json.load(f)[f"{prog}-{seed}"]
    harness.compare_fingerprint(want, port, f"fuzz {prog} seed {seed}: reference (stored fingerprint) vs port")
    if pyoracle.available("reference"):
        ref = harness.run_script(harness.OracleBackend("reference"), fuzz_script(prog, seed))
        harness.compare(ref, port, f"fuzz {prog} seed {seed}: reference vs port")


# Round-1 history: on the mutated pipeline corpus the device used to emit 7-8 surplus nat_log_rb records.  Cause (found
# with tools/diag_fuzz.py): on that box cudaHostGetDevicePointer() succeeds for PAGEABLE memory too (HMM), so both the
# "pinned" and the "pageable" variant went through the zero-copy header gather, whose 64-byte slots (a) cut the L4
# header off frames with long IPv4 options — the program then parsed, and rewrote, the NEXT frame's bytes — and (b)
# never wrote chunk 0 back, losing the port nat44_egress stores at bytes 14-15 of a frame whose ihl is 0.  Fixed in
# ctx.cu / hostio.cu (96-byte slots sized per frame from ihl, pinned-ness from cudaPointerGetAttributes); every
# program is now a plain pass on every seed, pinned and pageable.
@pytest.mark.gpu
@pytest.mark.parametrize("pinned", [False, True], ids=["pageable", "pinned"])
@pytest.mark.parametrize("seed", [11, 13, 17, 23])
@pytest.mark.parametrize("prog", sorted(TARGETS))
def test_gpu_mutated_frames_agree(prog, seed, pinned, ora_kind):
    if ora_kind == "none":
        pytest.fail("no oracle library present on this box")
    want = harness.run_script(harness.OracleBackend(ora_kind), fuzz_script(prog, seed))
    be = harness.GpuBackend(pinned=pinned)
    try:
        got = harness.run_script(be, fuzz_script(prog, seed))
    finally:
        be.close()
    harness.compare(want, got, f"fuzz {prog} seed {seed} ({'pinned' if pinned else 'pageable'}): {ora_kind} oracle vs gpu")
