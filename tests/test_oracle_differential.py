"""Differential tests beyond the committed goldens: the scenario generators are re-seeded and the plain-C port
(oracle/port.c) must agree bit for bit with the reference's own C on every new corpus — verdicts, rewritten bytes,
lengths, counters, table contents, event records.  The reference's results are pinned by their fingerprints
(tests/golden/fresh_corpora.json, written by tests/golden/make_golden.py); where the reference build (oracle/_ref)
is present the port is also compared with it directly.

The GPU-marked twin replays the same fresh corpora on the device against whichever oracle is present."""
import json
import os

import pytest

import harness
import scenarios
from oracle import pyoracle

SEEDS = [0x1001, 0x2002, 0x3003]
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fresh_corpora.json")

FRESH = {
    "antispoof": lambda s: scenarios.antispoof_script(seed=s, n_subs=37, n=2500),
    "qos": lambda s: scenarios.qos_script(seed=s, n_subs=29, n=3500),
    "nat": lambda s: scenarios.nat_script(seed=s, flags=0x0F, n_subs=17, pps=8, n=2000, name=f"nat_{s:x}"),
    "nat_parity_noeim": lambda s: scenarios.nat_script(seed=s, flags=0x2E, n_subs=11, pps=16, n=1500, name=f"natp_{s:x}"),
    "dhcp": lambda s: scenarios.dhcp_script(seed=s),
    "pipeline": lambda s: scenarios.pipeline_script(seed=s, n_subs=23, n=2500, flags=0x0F),
}

@pytest.mark.parametrize("seed", SEEDS)
@pytest.mark.parametrize("family", sorted(FRESH))
def test_port_agrees_with_reference_on_fresh_corpora(family, seed):
    port = harness.run_script(harness.OracleBackend("port"), FRESH[family](seed))
    with open(GOLD) as f:
        want = json.load(f)[f"{family}-{seed:#x}"]
    harness.compare_fingerprint(want, port, f"{family} seed {seed:#x}: reference (stored fingerprint) vs port")
    if pyoracle.available("reference"):
        ref = harness.run_script(harness.OracleBackend("reference"), FRESH[family](seed))
        harness.compare(ref, port, f"{family} seed {seed:#x}: reference vs port")


@pytest.mark.gpu
@pytest.mark.parametrize("seed", SEEDS[:2])
@pytest.mark.parametrize("family", sorted(FRESH))
def test_gpu_agrees_with_oracle_on_fresh_corpora(family, seed, ora_kind):
    if ora_kind == "none":
        pytest.fail("no oracle library present on this box")
    want = harness.run_script(harness.OracleBackend(ora_kind), FRESH[family](seed))
    be = harness.GpuBackend(pinned=bool(seed & 1))
    try:
        got = harness.run_script(be, FRESH[family](seed))
    finally:
        be.close()
    harness.compare(want, got, f"{family} seed {seed:#x}: {ora_kind} oracle vs gpu")
