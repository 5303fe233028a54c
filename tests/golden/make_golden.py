"""Generates tests/golden/*.npz by running every script of tests/scenarios.py
through the REFERENCE oracle (oracle/_ref/libbng_ref.so = the reference's own
eBPF C sources compiled natively), and the fingerprints (shape and SHA-256 per
result key) of the reference's results on the corpora of
tests/test_oracle_differential.py and tests/test_oracle_fuzz.py, which are too
large to store whole.  Needs the reference sources to (re)build that library;
the fixtures it writes are committed and travel.

    python tests/golden/make_golden.py              # everything
    python tests/golden/make_golden.py fingerprints # only the two .json files
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import harness  # noqa: E402
import scenarios  # noqa: E402
from oracle import pyoracle  # noqa: E402

FRESH_JSON = os.path.join(HERE, "fresh_corpora.json")
FUZZ_JSON = os.path.join(HERE, "mutated_frames.json")


def fresh_cases():
    """{case id: script factory} of test_oracle_differential's re-seeded corpora."""
    import test_oracle_differential as D
    return {f"{fam}-{seed:#x}": (lambda f=fam, s=seed: D.FRESH[f](s)) for fam in sorted(D.FRESH) for seed in D.SEEDS}


def fuzz_cases():
    """{case id: script factory} of test_oracle_fuzz's mutated corpora (the seeds the oracle-only test runs)."""
    import test_oracle_fuzz as F
    return {f"{prog}-{seed}": (lambda p=prog, s=seed: F.fuzz_script(p, s)) for prog in sorted(F.TARGETS) for seed in F.SEEDS}


def write_fingerprints(path, cases):
    out = {}
    for cid, fn in cases.items():
        out[cid] = harness.fingerprint(harness.run_script(harness.OracleBackend("reference"), fn()))
    with open(path, "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
        f.write("\n")
    print(f"{os.path.basename(path)}: {len(out)} cases, {os.path.getsize(path) / 1024:.0f} KiB")


def main():
    pyoracle.build("ref")
    if sys.argv[1:] != ["fingerprints"]:
        for name, fn in scenarios.ALL_SCRIPTS.items():
            be = harness.OracleBackend("reference")
            res = harness.run_script(be, fn())
            path = os.path.join(HERE, name + ".npz")
            harness.save_golden(path, res)
            print(f"{name}: {len(res)} arrays, {os.path.getsize(path) / 1024:.0f} KiB")
    write_fingerprints(FRESH_JSON, fresh_cases())
    write_fingerprints(FUZZ_JSON, fuzz_cases())


if __name__ == "__main__":
    main()
